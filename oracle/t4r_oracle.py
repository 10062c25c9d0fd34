"""CPU oracle for the session-sequence transformer hot path.

TEST INFRASTRUCTURE ONLY.  Nothing in ``transformers4rec_b200`` (the product) may
import this module; only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` do, and there only
as the checker / the CPU arm.

It is a plain-PyTorch (CPU, fp32) restatement of the reference's forward for
the path SURVEY.md §8a names.  Every function cites the reference file:line it
follows (paths relative to the upstream repo; ``HF:`` = the installed Hugging
Face ``transformers`` package, which owns the encoder arithmetic).

Pinning status (see DESIGN.md "Oracle"):
  * masking (MLM/CLM), LogUniformSampler, sampled/full-softmax head and RecallAt
    are pinned against the *reference's own code* executed in the authoring
    container (``tests/golden/make_golden.py`` loads the upstream files with
    stubbed third-party imports and records input/output vectors under
    ``tests/golden/``), and against the reference's known-answer tests
    (``tests/unit/torch/test_ranking_metrics.py:49-115``).
  * the encoders are pinned against the installed HF ``XLNetModel`` /
    ``GPT2Model`` built with the reference's kwargs
    (``transformers4rec/config/transformer.py:467-482`` / ``:244-260``); the
    reference's own tests hold shape checks only for that boundary, so encoder
    numerics are "parity unpinned by the reference" and pinned to HF instead.
"""
from __future__ import annotations

import math
from typing import Callable, Dict, Optional, Tuple

import torch
import torch.nn.functional as F

# --------------------------------------------------------------------------- #
# random draws: the reference consumes torch.bernoulli / torch.multinomial.
# Bit-exact parity is only defined for identical draws, so the oracle (and the
# golden generator, which monkey-patches torch.bernoulli/multinomial while it
# runs the upstream code) derive both from explicit uniforms.
# --------------------------------------------------------------------------- #


def bernoulli_from_uniform(u: torch.Tensor, p: float) -> torch.Tensor:
    """Stand-in for ``torch.bernoulli(full(p))``: 1 where u < p."""
    return (u < p)


def pick_kth_set(weights01: torch.Tensor, u: torch.Tensor) -> torch.Tensor:
    """Stand-in for ``torch.multinomial(weights01.float(), 1).squeeze()`` when
    the weights are 0/1: picks the k-th set position, k = min(floor(u*n), n-1).
    Rows with n == 0 return 0 (torch.multinomial would raise there)."""
    w = weights01.bool()
    n = w.sum(dim=1)
    k = torch.minimum((u.double() * n.double()).floor().long(), (n - 1).clamp(min=0))
    csum = w.long().cumsum(dim=1)  # 1-based rank at set positions
    hit = w & (csum == (k + 1).unsqueeze(1))
    idx = hit.float().argmax(dim=1)
    return torch.where(n > 0, idx, torch.zeros_like(idx))


# --------------------------------------------------------------------------- #
# ragged ingest (SURVEY §8f N1)
# --------------------------------------------------------------------------- #


def pad_ragged(values: torch.Tensor, offsets: torch.Tensor, padding_length: int) -> torch.Tensor:
    """utils/padding.py:48-68: ragged rows -> dense, right-padded with zeros, truncated to
    ``padding_length`` (the reference densifies a sparse COO tensor, then F.pad's it)."""
    rows = offsets.numel() - 1
    out = torch.zeros((rows, padding_length), dtype=values.dtype)
    for r in range(rows):
        seg = values[int(offsets[r]): int(offsets[r + 1])][:padding_length]
        out[r, : seg.numel()] = seg
    return out


def pad_dense(t: torch.Tensor, length: int) -> torch.Tensor:
    """utils/padding.py:20-30."""
    return F.pad(t, (0, length - t.shape[1], 0, 0)) if t.dim() == 2 else t


def pad_inputs(inputs: Dict[str, torch.Tensor], max_sequence_length: Optional[int] = None):
    """utils/padding.py:125-164 (+ pad_batch :71-122)."""
    batch_max = 0
    for k, v in inputs.items():
        if k.endswith("__offsets"):
            batch_max = max(int((v[1:] - v[:-1]).max()), batch_max)
    length = batch_max if max_sequence_length is None else min(max_sequence_length, batch_max)
    if length <= 0:
        return inputs
    out = {}
    for k, v in inputs.items():
        if k.endswith("__offsets"):
            col = k[: -len("__offsets")]
            out[col] = pad_ragged(inputs[col + "__values"], v, length)
        elif not k.endswith("__values"):
            out[k] = v
    return out


# --------------------------------------------------------------------------- #
# input block
# --------------------------------------------------------------------------- #


def embed_concat(
    tables: Dict[str, torch.Tensor],
    cat_inputs: Dict[str, torch.Tensor],
    cont_inputs: Optional[Dict[str, torch.Tensor]] = None,
    padding_idx: int = 0,
) -> torch.Tensor:
    """features/embedding.py:226-249 (per-feature ``nn.Embedding`` with
    ``padding_idx`` row, features/sequence.py:75-81), features/continuous.py:60-63
    (``unsqueeze(-1)``) and tabular/aggregation.py:35-47 (``torch.cat`` over
    *sorted* feature names)."""
    outs = {}
    for name, ids in cat_inputs.items():
        outs[name] = F.embedding(ids, tables[name], padding_idx=padding_idx)
    for name, val in (cont_inputs or {}).items():
        outs[name] = val.float().unsqueeze(-1)
    return torch.cat([outs[k] for k in sorted(outs.keys())], dim=-1)


def expand_non_sequential(features: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """tabular/base.py:53-63: features without a sequence axis ([B, dim]) are repeated
    over the L positions of the sequential ones."""
    seq = {k: v for k, v in features.items() if v.dim() >= 3}
    if not seq:
        return dict(features)
    L = next(iter(seq.values())).shape[1]
    return {k: (v if v.dim() >= 3 else v.unsqueeze(1).repeat(1, L, 1)) for k, v in features.items()}


def tabular_layer_norm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """tabular/transformations.py:95-141: ``nn.LayerNorm(dim)`` on one feature, before aggregation."""
    return F.layer_norm(x, (x.shape[-1],), gamma, beta, eps)


def soft_embedding(x: torch.Tensor, proj_weight: torch.Tensor, proj_bias: torch.Tensor,
                   table: torch.Tensor) -> torch.Tensor:
    """features/embedding.py:517-556 (SoftEmbedding.forward): ``softmax(Linear(1, n)(x))``
    weighted mean of the n embedding rows.  proj_weight [n, 1], proj_bias [n], table [n, dim]."""
    w = torch.softmax(F.linear(x.float().unsqueeze(-1), proj_weight, proj_bias), dim=-1)
    return (w.unsqueeze(-1) * table).sum(-2)


def aggregate(features: Dict[str, torch.Tensor], mode: str = "concat", item_name: Optional[str] = None) -> torch.Tensor:
    """tabular/aggregation.py:35-47 (concat), :139-157 (element-wise-sum), :160-193
    (element-wise-sum-item-multi); all iterate the features in sorted-name order."""
    feats = expand_non_sequential(features)
    names = sorted(feats.keys())
    if mode == "concat":
        return torch.cat([feats[n] for n in names], dim=-1)
    if len(set(v.shape for v in feats.values())) != 1:
        raise ValueError("The shapes of all input features are not equal, which is required for"
                         " element-wise aggregation: {}".format({k: v.shape for k, v in feats.items()}))
    if mode == "element-wise-sum":
        return torch.stack([feats[n] for n in names], dim=0).sum(dim=0)
    if mode == "element-wise-sum-item-multi":
        others = torch.stack([feats[n] for n in names if n != item_name], dim=0).sum(dim=0)
        return feats[item_name].multiply(others)
    raise ValueError(mode)


def stochastic_swap_noise(values: torch.Tensor, mask: Optional[torch.Tensor], u: torch.Tensor, perm: torch.Tensor,
                          replacement_prob: float) -> torch.Tensor:
    """tabular/transformations.py:54-92 (StochasticSwapNoise.augment, training mode) with the
    draws made explicit: ``u`` replaces ``torch.bernoulli`` (replace where u < p), ``perm``
    replaces ``torch.randperm(number of kept values)``."""
    if mask is not None and values.dim() == mask.dim() - 1:
        mask = mask[:, 0]
    rep = bernoulli_from_uniform(u, replacement_prob)
    if mask is not None:
        rep = rep & mask
    n_rep = int(rep.sum())
    pool = torch.masked_select(values, mask) if mask is not None else values.reshape(-1).clone()
    sampled = pool[perm][:n_rep]
    out = values.clone()
    out[rep] = sampled
    return out


def project_relu(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    """block/mlp.py:123-144: ``Linear`` + ``ReLU`` (the projection MLPBlock built at
    features/sequence.py:213-219)."""
    return F.relu(F.linear(x, weight, bias))


# --------------------------------------------------------------------------- #
# masking (integer, bit-exact)
# --------------------------------------------------------------------------- #


def predict_all(item_ids: torch.Tensor, padding_idx: int = 0):
    """masking.py:182-213."""
    labels = item_ids[:, 1:]
    labels = torch.cat([labels, torch.zeros((labels.shape[0], 1), dtype=labels.dtype)], dim=-1)
    mask_labels = labels != padding_idx
    return mask_labels, labels


def mlm_compute_masked_targets(
    item_ids: torch.Tensor,
    training: bool = False,
    testing: bool = False,
    padding_idx: int = 0,
    eval_on_last_item_seq_only: bool = True,
    mlm_probability: float = 0.15,
    u_bern: Optional[torch.Tensor] = None,
    u_force: Optional[torch.Tensor] = None,
    u_unmask: Optional[torch.Tensor] = None,
) -> Tuple[torch.Tensor, torch.Tensor]:
    """masking.py:376-470.  Returns (mask_schema bool [B,L(+1)], masked_targets i64)."""
    non_padded_mask = item_ids != padding_idx
    rows_ids = torch.arange(item_ids.size(0), dtype=torch.long)
    if not training and not testing:
        # masking.py:403-418 (inference: one extra [MASK] position)
        labels = torch.full((item_ids.shape[0], item_ids.shape[1] + 1), padding_idx, dtype=item_ids.dtype)
        last_item_sessions = non_padded_mask.sum(dim=1)
        labels[rows_ids, last_item_sessions] = item_ids[rows_ids, last_item_sessions - 1]
        return labels != padding_idx, labels

    labels = torch.full(item_ids.shape, padding_idx, dtype=item_ids.dtype)
    if training:
        # masking.py:424-459
        mask_labels = bernoulli_from_uniform(u_bern, mlm_probability) & non_padded_mask
        labels = torch.where(mask_labels, item_ids, torch.full_like(item_ids, padding_idx))
        one_random_index_by_session = pick_kth_set(non_padded_mask, u_force)
        labels[rows_ids, one_random_index_by_session] = item_ids[rows_ids, one_random_index_by_session]
        mask_labels = labels != padding_idx
        sequences_with_only_labels = mask_labels.sum(dim=1) == non_padded_mask.sum(dim=1)
        sampled_labels_to_unmask = pick_kth_set(mask_labels, u_unmask)
        labels_to_unmask = torch.masked_select(sampled_labels_to_unmask, sequences_with_only_labels)
        rows_to_unmask = torch.masked_select(rows_ids, sequences_with_only_labels)
        labels[rows_to_unmask, labels_to_unmask] = padding_idx
        mask_labels = labels != padding_idx
    else:
        # masking.py:461-468
        if eval_on_last_item_seq_only:
            last_item_sessions = non_padded_mask.sum(dim=1) - 1
            labels[rows_ids, last_item_sessions] = item_ids[rows_ids, last_item_sessions]
            mask_labels = labels != padding_idx
        else:
            mask_labels, labels = predict_all(item_ids, padding_idx)
    return mask_labels, labels


def mlm_apply_mask_to_inputs(x, mask_schema, masked_item_embedding, training=False, testing=False):
    """masking.py:473-498."""
    if not testing and not training:
        x = torch.cat([x, x[:, -1, :].unsqueeze(1)], dim=1)
    return torch.where(mask_schema.unsqueeze(-1).bool(), masked_item_embedding.to(x.dtype), x)


def clm_compute_masked_targets(
    item_ids: torch.Tensor,
    training: bool = False,
    testing: bool = False,
    padding_idx: int = 0,
    eval_on_last_item_seq_only: bool = True,
    train_on_last_item_seq_only: bool = False,
) -> Tuple[torch.Tensor, torch.Tensor]:
    """masking.py:274-300."""
    if not training and not testing:
        return item_ids != padding_idx, item_ids
    mask_labels, labels = predict_all(item_ids, padding_idx)
    if (eval_on_last_item_seq_only and not training) or (train_on_last_item_seq_only and training):
        rows_ids = torch.arange(labels.size(0), dtype=torch.long)
        last_item_sessions = mask_labels.sum(dim=1) - 1
        label_seq_trg_eval = torch.zeros(labels.shape, dtype=labels.dtype)
        label_seq_trg_eval[rows_ids, last_item_sessions] = labels[rows_ids, last_item_sessions]
        labels = label_seq_trg_eval
        mask_labels = item_ids != padding_idx
    return mask_labels, labels


def clm_apply_mask_to_inputs(x, mask_schema, masked_item_embedding, training=False, testing=False):
    """masking.py:302-337."""
    if not training and not testing:
        return torch.where(mask_schema.unsqueeze(-1).bool(), x, masked_item_embedding.to(x.dtype))
    pos_emb_inp = x[:, :-1]
    pos_emb_inp = torch.cat(
        [pos_emb_inp, torch.zeros((pos_emb_inp.shape[0], 1, pos_emb_inp.shape[2]), dtype=pos_emb_inp.dtype)], dim=1
    )
    return torch.where(mask_schema.unsqueeze(-1).bool(), pos_emb_inp, masked_item_embedding.to(pos_emb_inp.dtype))


def randint_from_uniform(u: float, n: int) -> int:
    """Stand-in for ``torch.randint(n, (1,)).item()``: min(floor(u * n), n - 1), in double like pick_kth_set."""
    return min(int(math.floor(float(u) * n)), n - 1)


def plm_context_lengths(max_span_length: int, plm_probability: float):
    """masking.py:608: ``int(span_length / plm_probability)`` for span_length = 0..max (index 0 unused)."""
    return [0] + [int(sp / plm_probability) for sp in range(1, max_span_length + 1)]


def plm_compute_masked_targets(item_ids: torch.Tensor, training: bool = False, padding_idx: int = 0,
                               eval_on_last_item_seq_only: bool = True, plm_probability: float = 1 / 6,
                               max_span_length: int = 5, permute_all: bool = False, draws: Optional[dict] = None):
    """masking.py:548-727 (PermutationLanguageModeling._compute_masked_targets_extended).

    Returns (mask_labels bool [B,L], labels i64 [B,L], target_mapping f32 [B,L,L], perm_mask [B,L,L] (f32 in
    training, i64 in evaluation, like the reference), info) where ``info`` records how many draws each session
    consumed (the golden generator needs it to line the upstream code's sequential draws up with these
    per-session ones).

    Draws (training; the reference calls torch.randint twice per loop iteration, torch.multinomial and
    torch.randperm): ``u_span`` / ``u_start`` [B, NMAX] uniforms for the span length / start offset of iteration
    n of session b (span = 1 + floor(u*max_span), start = cur_len + floor(u*(context - span + 1))), ``u_force``
    [B] (one position when nothing got masked), ``u_unmask`` [B] (one label removed when everything is a label),
    ``perm`` [B, L] the factorisation order (a permutation of 0..L-1 per session)."""
    B, L = item_ids.shape
    labels = torch.full(item_ids.shape, padding_idx, dtype=item_ids.dtype)
    non_padded_mask = item_ids != padding_idx
    rows_ids = torch.arange(B, dtype=torch.long)
    mask_labels = torch.zeros(labels.shape, dtype=torch.bool)
    info = {"n_iter": [0] * B, "forced": [False] * B}
    if training:
        target_mapping = torch.zeros((B, L, L), dtype=torch.float32)
        perm_mask = torch.zeros((B, L, L), dtype=torch.float32)
        ctx = plm_context_lengths(max_span_length, plm_probability)
        if permute_all:
            mask_labels = non_padded_mask.clone()
        else:
            for i in range(B):
                cur_len, n = 0, 0
                max_len = int(non_padded_mask[i].sum())
                while cur_len < max_len:
                    span_length = 1 + randint_from_uniform(draws["u_span"][i, n], max_span_length)
                    context_length = ctx[span_length]
                    start_index = cur_len + randint_from_uniform(draws["u_start"][i, n], context_length - span_length + 1)
                    if start_index < max_len:
                        mask_labels[i, start_index: start_index + span_length] = True
                    cur_len += context_length
                    n += 1
                info["n_iter"][i] = n
                if mask_labels[i].sum() == 0:
                    k = pick_kth_set(non_padded_mask[i: i + 1], draws["u_force"][i: i + 1])[0]
                    mask_labels[i, k] = bool(item_ids[i, k] != 0)  # the reference assigns the item id into a bool tensor
                    info["forced"][i] = True
                target_mapping[i] = torch.eye(L)
        labels = torch.where(mask_labels, item_ids, torch.full_like(item_ids, padding_idx))
        sequences_with_only_labels = mask_labels.sum(dim=1) == non_padded_mask.sum(dim=1)
        sampled_labels_to_unmask = pick_kth_set(mask_labels, draws["u_unmask"])
        labels_to_unmask = torch.masked_select(sampled_labels_to_unmask, sequences_with_only_labels)
        rows_to_unmask = torch.masked_select(rows_ids, sequences_with_only_labels)
        labels[rows_to_unmask, labels_to_unmask] = padding_idx
        mask_labels = labels != padding_idx
        for i in range(B):
            perm_index = draws["perm"][i].long().clone()          # arange(L)[randperm(L)]
            perm_index.masked_fill_(~mask_labels[i], -1)
            perm_mask[i] = ((perm_index.reshape((L, 1)) <= perm_index.reshape((1, L))) & mask_labels[i]).float()
    else:
        causal = torch.triu(torch.ones([L, L]), diagonal=1)
        if eval_on_last_item_seq_only:
            last_item_sessions = non_padded_mask.sum(dim=1) - 1
            labels[rows_ids, last_item_sessions] = item_ids[rows_ids, last_item_sessions]
            mask_labels = labels != padding_idx
            perm_mask = torch.zeros((B, L, L), dtype=torch.float32)
            perm_mask[rows_ids, :, last_item_sessions] = 1
            perm_mask = ((causal.expand((B, L, L)) + perm_mask) > 0).long()
            target_mapping = torch.diag(torch.ones(L, dtype=torch.float32)).expand((B, L, L))
        else:
            mask_labels, labels = predict_all(item_ids, padding_idx)
            target_mapping = F.one_hot(torch.arange(0, L, dtype=torch.long), num_classes=L).expand((B, L, L))
            perm_mask = ((causal.expand((B, L, L)) + torch.zeros((B, L, L))) > 0).long()
    return mask_labels, labels, target_mapping, perm_mask, info


def plm_apply_mask_to_inputs(x, mask_schema, masked_item_embedding, training=False, testing=False):
    """masking.py:155-180 (the base-class rule PLM inherits): nothing at inference."""
    if not training and not testing:
        return x
    return torch.where(mask_schema.unsqueeze(-1).bool(), masked_item_embedding.to(x.dtype), x)


def hf_encoder_forward_plm(model, x: torch.Tensor, perm_mask: torch.Tensor, target_mapping: torch.Tensor) -> torch.Tensor:
    """block/transformer.py:179-199 with masking.transformer_arguments = {target_mapping, perm_mask} (masking.py:739-740):
    HF returns the query stream g (one row per target position) as output[0]."""
    return model(inputs_embeds=x, perm_mask=perm_mask.to(x.dtype), target_mapping=target_mapping.to(x.dtype))[0]


# --------------------------------------------------------------------------- #
# encoders: (1) the installed HF models built with the reference's kwargs,
#           (2) a literal restatement of the math (SURVEY Appendix A) used as
#               the kernel contract and cross-checked against (1) in tests.
# --------------------------------------------------------------------------- #


def build_hf_xlnet(d_model: int, n_head: int, n_layer: int, **kw):
    """config/transformer.py:467-482 (XLNetConfig.build) + :67-69 (MODEL_MAPPING)."""
    import transformers

    cfg = transformers.XLNetConfig(
        d_model=d_model,
        d_inner=d_model * 4,
        n_layer=n_layer,
        n_head=n_head,
        attn_type="bi",
        ff_activation="gelu",
        initializer_range=0.01,
        layer_norm_eps=0.03,
        dropout=0.3,
        pad_token_id=0,
        output_attentions=False,
        vocab_size=1,
        mem_len=1,
        **kw,
    )
    return transformers.XLNetModel(cfg)


def build_hf_gpt2(d_model: int, n_head: int, n_layer: int, total_seq_length: int, **kw):
    """config/transformer.py:244-260 (GPT2Config.build).  ``layer_norm_eps`` is passed
    under a name HF's GPT2Config does not read, so the effective LN eps is HF's
    default 1e-5 (SURVEY §7 quirk 8)."""
    import transformers

    cfg = transformers.GPT2Config(
        n_embd=d_model,
        n_inner=d_model * 4,
        n_layer=n_layer,
        n_head=n_head,
        activation_function="gelu",
        initializer_range=0.01,
        layer_norm_eps=0.03,
        resid_pdrop=0.3,
        embd_pdrop=0.3,
        attn_pdrop=0.3,
        n_positions=total_seq_length,
        n_ctx=total_seq_length,
        output_attentions=False,
        vocab_size=1,
        **kw,
    )
    return transformers.GPT2Model(cfg)


def hf_encoder_forward(model, x: torch.Tensor) -> torch.Tensor:
    """block/transformer.py:179-199: call HF with ``inputs_embeds`` only, take output[0]."""
    return model(inputs_embeds=x)[0]


def xlnet_relative_positions(L: int, d: int) -> torch.Tensor:
    """HF:models/xlnet/modeling_xlnet.py:930-976 for attn_type='bi', bi_data=False,
    clamp_len=-1: positions klen..-qlen+1 (klen == qlen == L, no mems fed back),
    sin || cos (not interleaved).  Returns [2L, d]."""
    freq_seq = torch.arange(0, d, 2.0, dtype=torch.float32)
    inv_freq = 1.0 / torch.pow(10000, (freq_seq / d))
    pos_seq = torch.arange(L, -L, -1.0, dtype=torch.float32)
    sinusoid = torch.einsum("i,d->id", pos_seq, inv_freq)
    return torch.cat([torch.sin(sinusoid), torch.cos(sinusoid)], dim=-1)


def xlnet_forward_restated(x: torch.Tensor, sd: Dict[str, torch.Tensor], n_layer: int, n_head: int,
                           eps: float = 0.03, drop=None) -> torch.Tensor:
    """Literal restatement of HF XLNetModel.forward for the arguments the reference
    passes (inputs_embeds only; HF:xlnet:979-1205, rel_attn_core :95-140,
    rel_shift_bnij :81-93, post_attention :142-152, XLNetFeedForward :285-305).
    x: [B, L, d] -> [B, L, d].  ``sd`` uses HF state_dict names.

    ``drop(site, tensor)`` (train mode; None = eval) is called at every place HF applies ``self.dropout``: site 0 the
    input rows (:1085), 5 the returned rows (:1180); per layer l, base 16 (l + 1): +1 the attention probabilities
    [B, H, L, L] (:129), +2 the output projection (:147), +3 after the activation (:300), +4 after layer_2 (:302).
    Site base + 0 is the projected relative-position table [2L, d]: HF drops pos_emb [2L, B, d] per batch element
    before projecting it (:1159); the product drops the shared projection instead (DESIGN: dropout) -- with ``drop``
    returning its argument at that site the function is HF's."""
    B, L, d = x.shape
    H = n_head
    dh = d // H
    pos = xlnet_relative_positions(L, d).to(x.dtype)  # [2L, d]
    scale = 1.0 / math.sqrt(dh)
    D = drop if drop is not None else (lambda site, t: t)
    h = D(0, x)
    for i in range(n_layer):
        s0 = 16 * (i + 1)
        p = f"layer.{i}."
        Wq = sd[p + "rel_attn.q"].reshape(d, H * dh)
        Wk = sd[p + "rel_attn.k"].reshape(d, H * dh)
        Wv = sd[p + "rel_attn.v"].reshape(d, H * dh)
        Wo = sd[p + "rel_attn.o"].reshape(d, H * dh)
        Wr = sd[p + "rel_attn.r"].reshape(d, H * dh)
        rw = sd[p + "rel_attn.r_w_bias"]  # [H, dh]
        rr = sd[p + "rel_attn.r_r_bias"]
        q = (h @ Wq).view(B, L, H, dh)
        k = (h @ Wk).view(B, L, H, dh)
        v = (h @ Wv).view(B, L, H, dh)
        r = D(s0, pos @ Wr).view(2 * L, H, dh)
        ac = torch.einsum("bihd,bjhd->bhij", q + rw, k)
        bd_full = torch.einsum("bihd,mhd->bhim", q + rr, r)  # [B,H,L,2L]
        # rel_shift_bnij identity: shift(x)[i, j] == x[i, j + L - i]
        idx = (torch.arange(L).view(1, L) + L - torch.arange(L).view(L, 1))  # [L(i), L(j)]
        bd = torch.gather(bd_full, 3, idx.view(1, 1, L, L).expand(B, H, L, L))
        prob = D(s0 + 1, torch.softmax((ac + bd) * scale, dim=-1))
        a = torch.einsum("bhij,bjhd->bihd", prob, v).reshape(B, L, H * dh)
        attn_out = D(s0 + 2, a @ Wo.t())
        h = F.layer_norm(h + attn_out, (d,), sd[p + "rel_attn.layer_norm.weight"], sd[p + "rel_attn.layer_norm.bias"], eps)
        ff = F.linear(h, sd[p + "ff.layer_1.weight"], sd[p + "ff.layer_1.bias"])
        ff = D(s0 + 3, F.gelu(ff))
        ff = D(s0 + 4, F.linear(ff, sd[p + "ff.layer_2.weight"], sd[p + "ff.layer_2.bias"]))
        h = F.layer_norm(h + ff, (d,), sd[p + "ff.layer_norm.weight"], sd[p + "ff.layer_norm.bias"], eps)
    return D(5, h)


def gpt2_forward_restated(x: torch.Tensor, sd: Dict[str, torch.Tensor], n_layer: int, n_head: int,
                          eps: float = 1e-5, drop=None) -> torch.Tensor:
    """Literal restatement of HF GPT2Model.forward with inputs_embeds only
    (HF:models/gpt2/modeling_gpt2.py:522-636, GPT2Block :246-309, GPT2Attention
    :144-226, GPT2MLP :229-243).  Conv1D weights are [in, out] (y = x @ W + b).
    ``drop(site, tensor)`` marks HF's dropout calls (train mode): 0 after the position embeddings (:584), per layer l,
    base 16 (l + 1): +1 the attention probabilities [B, H, L, L] (:66), +2 the attention output projection (:225),
    +4 the MLP output projection (:241)."""
    B, L, d = x.shape
    H = n_head
    dh = d // H
    D = drop if drop is not None else (lambda site, t: t)
    h = D(0, x + sd["wpe.weight"][:L].unsqueeze(0))
    causal = torch.tril(torch.ones(L, L, dtype=torch.bool))
    for i in range(n_layer):
        s0 = 16 * (i + 1)
        p = f"h.{i}."
        a = F.layer_norm(h, (d,), sd[p + "ln_1.weight"], sd[p + "ln_1.bias"], eps)
        qkv = a @ sd[p + "attn.c_attn.weight"] + sd[p + "attn.c_attn.bias"]
        q, k, v = qkv.split(d, dim=-1)
        q = q.view(B, L, H, dh).transpose(1, 2)
        k = k.view(B, L, H, dh).transpose(1, 2)
        v = v.view(B, L, H, dh).transpose(1, 2)
        s = (q @ k.transpose(-1, -2)) / math.sqrt(dh)
        s = s.masked_fill(~causal, float("-inf"))
        o = (D(s0 + 1, torch.softmax(s, dim=-1)) @ v).transpose(1, 2).reshape(B, L, d)
        h = h + D(s0 + 2, o @ sd[p + "attn.c_proj.weight"] + sd[p + "attn.c_proj.bias"])
        m = F.layer_norm(h, (d,), sd[p + "ln_2.weight"], sd[p + "ln_2.bias"], eps)
        m = F.gelu(m @ sd[p + "mlp.c_fc.weight"] + sd[p + "mlp.c_fc.bias"])
        h = h + D(s0 + 4, m @ sd[p + "mlp.c_proj.weight"] + sd[p + "mlp.c_proj.bias"])
    return F.layer_norm(h, (d,), sd["ln_f.weight"], sd["ln_f.bias"], eps)


# --------------------------------------------------------------------------- #
# head
# --------------------------------------------------------------------------- #


def remove_pad_3d(x: torch.Tensor, non_pad_mask: torch.Tensor) -> torch.Tensor:
    """model/prediction_task.py:472-479."""
    x = x.flatten(end_dim=1)
    fl = torch.masked_select(x, non_pad_mask.unsqueeze(1).expand_as(x))
    return fl.view(-1, x.size(1))


def select_targets(x: torch.Tensor, masked_targets: torch.Tensor, padding_idx: int = 0):
    """model/prediction_task.py:436-443: flatten labels, keep non-pad, compact rows."""
    trg_flat = masked_targets.flatten()
    non_pad_mask = trg_flat != padding_idx
    y = torch.masked_select(trg_flat, non_pad_mask).long()
    return remove_pad_3d(x, non_pad_mask), y


def full_softmax_head(x_t: torch.Tensor, y: torch.Tensor, out_weight: torch.Tensor,
                      softmax_temperature: float = 1.0, label_smoothing: float = 0.0):
    """model/prediction_task.py:648-671 (logits = x @ W.T, optional temperature) and
    :446 / :347 (``nn.CrossEntropyLoss`` mean reduction; label smoothing per
    losses.py:4-20).  Returns (loss, logits)."""
    logits = x_t @ out_weight.t()
    if softmax_temperature:
        logits = torch.div(logits, softmax_temperature)
    loss = F.cross_entropy(logits, y, label_smoothing=label_smoothing)
    return loss, logits


def log_uniform_distr(max_id: int, min_id: int = 0) -> torch.Tensor:
    """model/prediction_task.py:766-787."""
    log_indices = torch.arange(1.0, max_id - min_id + 2.0, 1.0).log_()
    probs = (log_indices[1:] - log_indices[:-1]) / log_indices[-1]
    if min_id > 0:
        probs = torch.cat([torch.zeros([min_id], dtype=probs.dtype), probs], dim=0)
    return probs


def unique_sampling_distr(dist: torch.Tensor, n_sample: int) -> torch.Tensor:
    """model/prediction_task.py:789-796."""
    return (-(-dist.double().log1p_() * n_sample).expm1_()).float()


def negatives_from_draws(raw_draws: torch.Tensor, max_n_samples: int) -> torch.Tensor:
    """model/prediction_task.py:843-845: ``multinomial(dist, 2*S, replacement=True)
    .unique()[:S]`` -- sorted ascending, then truncated.  ``raw_draws`` are the
    multinomial's output ids (the random part)."""
    return raw_draws.unique()[:max_n_samples]


def sampled_softmax_head(x_t: torch.Tensor, y: torch.Tensor, out_weight: torch.Tensor,
                         neg_samples: torch.Tensor, unique_dist: torch.Tensor,
                         softmax_temperature: float = 1.0):
    """model/prediction_task.py:673-696 (+ :666-669 temperature, :446 CE)."""
    targets_probs = unique_dist[y]
    samples_probs = unique_dist[neg_samples]
    positive_weights = out_weight[y]
    negative_weights = out_weight[neg_samples]
    positive_scores = (x_t * positive_weights).sum(dim=-1, keepdim=True)
    negative_scores = x_t @ negative_weights.t()
    epsilon = 1e-16
    positive_scores = positive_scores - torch.unsqueeze(torch.log(targets_probs + epsilon), dim=-1)
    negative_scores = negative_scores - torch.unsqueeze(torch.log(samples_probs + epsilon), dim=0)
    accidental_hits = torch.unsqueeze(y, -1) == torch.unsqueeze(neg_samples, 0)
    negative_scores[accidental_hits] = torch.finfo(torch.float16).min / 100.0
    logits = torch.cat([positive_scores, negative_scores], dim=1)
    new_targets = torch.zeros(logits.shape[0], dtype=torch.int64)
    if softmax_temperature:
        logits = torch.div(logits, softmax_temperature)
    loss = F.cross_entropy(logits, new_targets)
    return loss, logits


def recall_at(ks, scores: torch.Tensor, labels: torch.Tensor, labels_onehot: bool = True) -> torch.Tensor:
    """ranking_metric.py:111-147 (+ utils/torch_utils.py:226-238).  ``labels`` are
    class ids when ``labels_onehot`` (the NextItemPredictionTask default), else a
    0/1 relevance matrix.  Returns per-row recalls [T, len(ks)]."""
    if labels_onehot:
        labels = F.one_hot(labels.reshape(-1).long(), scores.size(-1)).float()
    scores = scores.view(-1, scores.size(-1))
    labels = labels.view(-1, labels.size(-1))
    max_k = int(max(ks))
    _, topk_indices = torch.topk(scores, max_k)
    topk_labels = torch.gather(labels, 1, topk_indices)
    recalls = torch.zeros(scores.shape[0], len(ks), dtype=torch.float32)
    num_relevant = torch.sum(labels, dim=-1)
    rel_indices = (num_relevant != 0).nonzero().squeeze(dim=1)
    rel_count = num_relevant[rel_indices]
    if rel_indices.shape[0] > 0:
        for index, k in enumerate(ks):
            rel_labels = topk_labels[rel_indices, : int(k)]
            recalls[rel_indices, index] = torch.div(torch.sum(rel_labels, dim=-1), rel_count).to(torch.float32)
    return recalls


def recall_at_mean(ks, scores, labels, labels_onehot=True) -> torch.Tensor:
    """ranking_metric.py:52-63: one update = mean over rows of the batch."""
    return recall_at(ks, scores, labels, labels_onehot).mean(0)


def _topk_labels(ks, scores: torch.Tensor, labels: torch.Tensor, labels_onehot: bool):
    """utils/torch_utils.py:226-238 (extract_topk / tranform_label_to_onehot)."""
    if labels_onehot:
        labels = F.one_hot(labels.reshape(-1).long(), scores.size(-1)).float()
    scores = scores.view(-1, scores.size(-1))
    labels = labels.view(-1, labels.size(-1)).float()
    topk_scores, topk_indices = torch.topk(scores, int(max(ks)))
    return topk_scores, torch.gather(labels, 1, topk_indices), labels


def precision_at(ks, scores, labels, labels_onehot=True) -> torch.Tensor:
    """ranking_metric.py:73-103."""
    _, tl, _ = _topk_labels(ks, scores, labels, labels_onehot)
    return torch.stack([tl[:, : int(k)].sum(dim=1) / float(k) for k in ks], dim=1)


def avg_precision_at(ks, scores, labels, labels_onehot=True) -> torch.Tensor:
    """ranking_metric.py:150-190."""
    _, tl, lab = _topk_labels(ks, scores, labels, labels_onehot)
    max_k = int(max(ks))
    prec = torch.stack([tl[:, :j].sum(dim=1) / float(j) for j in range(1, max_k + 1)], dim=1)
    rel = prec * tl
    num_relevant = lab.sum(dim=1)
    return torch.stack([rel[:, : int(k)].sum(dim=1) / num_relevant.clamp(min=1, max=int(k)) for k in ks], dim=1)


def dcg_at(ks, scores, labels, labels_onehot=True, log_base: int = 2) -> torch.Tensor:
    """ranking_metric.py:193-238."""
    _, tl, _ = _topk_labels(ks, scores, labels, labels_onehot)
    pos = torch.arange(int(max(ks)), dtype=torch.float32)
    base = torch.log(torch.tensor([float(log_base)])).item()
    disc = 1 / (torch.log(pos + 2) / base)
    return torch.stack([(tl[:, : int(k)] * disc[: int(k)]).sum(dim=1) for k in ks], dim=1)


def ndcg_at(ks, scores, labels, labels_onehot=True) -> torch.Tensor:
    """ranking_metric.py:241-281: DCG of the ranking / DCG of the ideal ranking."""
    ts, tl, _ = _topk_labels(ks, scores, labels, labels_onehot)
    gains = dcg_at(ks, ts, tl, labels_onehot=False)
    ideal = dcg_at(ks, tl, tl, labels_onehot=False)
    return torch.where(ideal != 0, gains / ideal.clamp(min=1e-30), torch.zeros_like(gains))


def mrr_at(ks, scores, labels, labels_onehot=True) -> torch.Tensor:
    """ranking_metric.py:284-319."""
    _, tl, _ = _topk_labels(ks, scores, labels, labels_onehot)
    return torch.stack([(tl[:, : int(k)] / (torch.arange(int(k)) + 1)).max(dim=1).values for k in ks], dim=1)


# --------------------------------------------------------------------------- #
# end-to-end oracle (also the CPU baseline "module graph")
# --------------------------------------------------------------------------- #


class OracleSessionModel(torch.nn.Module):
    """The reference's module graph for one config of SURVEY §8d, restated with
    stock torch modules + the HF encoder: Model.forward (model/base.py:544-580) ->
    Head.forward (:371-407) -> SequentialBlock(TabularSequenceFeatures,
    TransformerBlock) -> NextItemPredictionTask.forward (prediction_task.py:419-451).
    """

    def __init__(self, *, cardinalities: Dict[str, int], embedding_dims: Dict[str, int], item_id: str,
                 continuous: Tuple[str, ...] = (), d_model: int, n_head: int, n_layer: int,
                 max_seq_len: int, arch: str = "xlnet", masking: str = "mlm",
                 project: bool = True, weight_tying: bool = True, sampled_softmax: bool = False,
                 max_n_samples: int = 100, softmax_temperature: float = 1.0, mlm_probability: float = 0.15):
        super().__init__()
        self.item_id = item_id
        self.continuous = tuple(continuous)
        self.masking = masking
        self.arch = arch
        self.mlm_probability = mlm_probability
        self.plm_kwargs: dict = {}      # plm_probability / max_span_length / eval_on_last_item_seq_only overrides
        self._plm = None
        self.softmax_temperature = softmax_temperature
        self.sampled_softmax = sampled_softmax
        self.max_n_samples = max_n_samples
        self.tables = torch.nn.ModuleDict()
        for name, card in cardinalities.items():
            emb = torch.nn.Embedding(card, embedding_dims[name], padding_idx=0)
            torch.nn.init.normal_(emb.weight, mean=0.0, std=0.05)  # features/embedding.py:461-462
            self.tables[name.replace("/", "__")] = emb
        self.table_names = list(cardinalities.keys())
        C = sum(embedding_dims.values()) + len(self.continuous)
        self.proj = torch.nn.Linear(C, d_model) if project else None
        hidden = d_model if project else C
        assert hidden == d_model
        self.masked_item_embedding = torch.nn.Parameter(torch.empty(hidden))
        torch.nn.init.normal_(self.masked_item_embedding, mean=0, std=0.001)  # masking.py:103-108
        if arch == "xlnet":
            self.transformer = build_hf_xlnet(d_model, n_head, n_layer)
        else:
            self.transformer = build_hf_gpt2(d_model, n_head, n_layer, max_seq_len)
        item_dim = embedding_dims[item_id]
        assert weight_tying
        # prediction_task.py:390-397: Linear(d -> item_dim), no activation, when dims differ
        self.task_block = torch.nn.Linear(d_model, item_dim) if d_model != item_dim else None
        self.V = cardinalities[item_id]
        if sampled_softmax:
            dist = log_uniform_distr(self.V, 1)
            self.register_buffer("dist", dist)
            self.register_buffer("unique_dist", unique_sampling_distr(dist, 2 * max_n_samples))

    def item_table(self) -> torch.Tensor:
        return self.tables[self.item_id.replace("/", "__")].weight

    def input_block(self, inputs, training, testing, draws=None):
        tables = {n: self.tables[n.replace("/", "__")].weight for n in self.table_names}
        x = embed_concat(tables, {n: inputs[n] for n in self.table_names},
                         {n: inputs[n] for n in self.continuous})
        if self.proj is not None:
            x = project_relu(x, self.proj.weight, self.proj.bias)
        ids = inputs[self.item_id]
        if self.masking == "mlm":
            d = draws or {}
            mask, labels = mlm_compute_masked_targets(ids, training, testing, mlm_probability=self.mlm_probability,
                                                      u_bern=d.get("u_bern"), u_force=d.get("u_force"),
                                                      u_unmask=d.get("u_unmask"))
            x = mlm_apply_mask_to_inputs(x, mask, self.masked_item_embedding, training, testing)
        elif self.masking == "plm":
            # masking.py:729-740: PLM's compute_masked_targets only looks at `training`
            mask, labels, tm, pm, _ = plm_compute_masked_targets(ids, training, draws=draws, **self.plm_kwargs)
            self._plm = (pm, tm)
            x = plm_apply_mask_to_inputs(x, mask, self.masked_item_embedding, training, testing)
        else:
            mask, labels = clm_compute_masked_targets(ids, training, testing)
            x = clm_apply_mask_to_inputs(x, mask, self.masked_item_embedding, training, testing)
        return x, mask, labels

    def forward(self, inputs, training=True, testing=False, draws=None, neg_samples=None):
        x, mask, labels = self.input_block(inputs, training, testing, draws)
        if self.masking == "plm":
            h = hf_encoder_forward_plm(self.transformer, x, *self._plm)   # output[0] = the query stream g
        else:
            h = hf_encoder_forward(self.transformer, x)
        hs = h
        if self.task_block is not None:
            h = self.task_block(h.to(self.task_block.weight.dtype))
        x_t, y = select_targets(h, labels)
        W = self.item_table()
        if self.sampled_softmax and training:
            loss, logits = sampled_softmax_head(x_t, y, W, neg_samples, self.unique_dist, self.softmax_temperature)
        else:
            loss, logits = full_softmax_head(x_t, y, W, self.softmax_temperature)
        # Head.forward :404-407 and Model.forward :574-576 reduce a 1-element stack by mean
        return {"loss": loss, "labels": y, "predictions": logits, "hidden": hs,
                "mask_schema": mask, "masked_targets": labels, "x_t": x_t}
