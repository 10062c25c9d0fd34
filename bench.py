#!/usr/bin/env python
"""bench.py -- sessions/sec (forward + loss) of the session-transformer hot path.

Contract: ``python bench.py --gpus N --steps K --warmup W`` (N>1 via torchrun, one
rank per GPU) prints ONE JSON line from rank 0.  A "step" is one pass of the hot
path (gather -> projection -> masking -> encoder -> tied-weight softmax CE) over one
batch of synthetic yoochoose-shaped sessions.  Workload at every N: BASELINE.json
configs[1] (1M-item table, L=20, XLNet d=256 x4, MLM, B=2048 per GPU; weak scaling,
independent replicas -- sessions are independent, no data-path collective).  After the
headline, every N also times the ROW-SHARDED table + tied head of configs[3] and configs[4]
(SURVEY 8e) and reports them in the line's ``sharded`` record.

``--impl reference`` times the reference's own CPU implementation of the path (the
oracle graph: stock torch ops + the Hugging Face encoder, all host threads) on a
bounded sample of the same workload.

``--dump-outputs DIR`` writes what the timed path returned in its last timed step as
``DIR/<name>.npy`` (see ``dump_outputs``).  Inputs, weights and random draws are seeded, so
two builds run with the same arguments can be compared output for output.

The benchmark writes nothing into the source tree (which may be read-only): no bytecode
caches, and its one scratch file goes to the system's temporary directory.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

SIDE6 = {"category/list": 337, "brand/list": 1000, "shop/list": 10000, "price_bin/list": 100, "weekday/list": 32,
         "hour_bin/list": 7}  # SURVEY §8d config 3: side cardinalities, all De = 64 (features/embedding.py:108)

CONFIGS = {
    # BASELINE.json configs[1] as instantiated in SURVEY.md §8d
    "config2": dict(V=1_000_001, De=256, d=256, H=8, NL=4, L=20, B=2048, arch="xlnet", masking="mlm",
                    label="1M-item table, seq_len=20, XLNet-base d_model=256 4-layer, MLM, batch=2048"),
    # BASELINE.json configs[2]: 7 categorical features (De = 64 each) -> concat 448 -> Linear(448 -> 256) + ReLU ->
    # CLM -> GPT-2 -> task_block Linear(256 -> 64) -> tied logits over the 64-d item table.  `--workload config3`.
    "config3": dict(V=1_000_001, De=64, d=256, H=8, NL=4, L=20, B=4096, arch="gpt2", masking="clm", side=SIDE6,
                    label="1M-item table + 6 categorical side features, ConcatFeatures aggregation, GPT-2 CLM, "
                          "batch=4096"),
    # BASELINE.json configs[4] at ONE rank's shard of the 50M-row table (6.25M rows), replicated -- the single-GPU
    # shape of that config (sampled softmax, 50K negatives, L=50).  `--workload config5`.
    "config5": dict(V=6_250_001, De=256, d=256, H=8, NL=4, L=50, B=2048, arch="xlnet", masking="mlm", sampled=50_000,
                    label="one rank's shard (6.25M rows) of the 50M-item table, sampled softmax 50K negatives, "
                          "seq_len=50, XLNet-base d_model=256 4-layer, MLM, batch=2048"),
    # BASELINE.json configs[0] (the reference's own CPU-runnable case); used by --workload config1
    "config1": dict(V=10_001, De=64, d=64, H=4, NL=2, L=20, B=512, arch="xlnet", masking="mlm",
                    label="synthetic yoochoose schema, 10K-item table, seq_len=20, XLNet d_model=64 2-layer"),
    # BASELINE.json configs[3]: the item table (= tied output layer) row-sharded over the ranks (SURVEY §8e);
    # one all-to-all on the lookup, one all-gather of (lse, label-logit) pairs on the head.  Parity-test case and
    # scaling probe (`--workload config4 --gpus N`), not the default bench line.
    "config4": dict(V=10_000_001, De=256, d=256, H=8, NL=4, L=20, B=2048, arch="xlnet", masking="mlm", sharded=True,
                    label="10M-item table row-sharded, tied-weight full softmax, XLNet-base d_model=256 4-layer, MLM, "
                          "batch=2048 per GPU"),
}
METRIC = "sessions/sec (fwd+loss)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def head_traffic(resident=True):
    """dram__bytes_read.sum + dram__bytes_write.sum of the head GEMM from the committed ncu capture
    (profiles/r2_head_traffic.json for the resident-A kernel, r1c_head_traffic.json for the streaming one; config2
    only) -- None when no capture is on record."""
    p = os.path.join(ROOT, "profiles", "r2_head_traffic.json" if resident else "r1c_head_traffic.json")
    try:
        with open(p) as f:
            return json.load(f)["dram_bytes_per_launch"]
    except Exception:
        return None


def ncu_tensor_pipe():
    """Per-kernel tensor-pipe utilisation from the committed ncu captures (profiles/r2_tensor_pipe.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_tensor_pipe.json")) as f:
            return json.load(f)
    except Exception:
        return None


def cardinalities(cfg):
    cards = {"item_id/list": cfg["V"]}
    for name, card in cfg.get("side", {}).items():
        cards[name] = card
    return cards


def synth_batch(B, L, cfg, seed=0):
    """Right-padded sessions, len ~ U{2..L}, ids uniform in [1, card) for every categorical feature (SURVEY §8d)."""
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(2, L + 1, (B,), generator=g)
    valid = torch.arange(L).unsqueeze(0) < lens.unsqueeze(1)
    out = {}
    for name, card in cardinalities(cfg).items():
        ids = torch.randint(1, card, (B, L), generator=g)
        out[name] = torch.where(valid, ids, torch.zeros_like(ids))
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_product_model(cfg, device, dropout=None):
    import transformers4rec_b200.torch as tr

    torch.manual_seed(1)
    cards = cardinalities(cfg)
    schema = tr.Schema([tr.ColumnSchema.create_categorical(n, c - 1, tags=[tr.Tags.ITEM_ID] if n == "item_id/list" else None)
                        for n, c in cards.items()])
    extra = dict(shard_item_table=True, device=device) if cfg.get("sharded") else {}  # allocate only this rank's rows
    inputs = tr.TabularSequenceFeatures.from_schema(schema, max_sequence_length=cfg["L"], d_output=cfg["d"],
                                                    masking=cfg["masking"],
                                                    embedding_dims={n: cfg["De"] for n in cards}, **extra)
    tcfg = (tr.XLNetConfig if cfg["arch"] == "xlnet" else tr.GPT2Config).build(
        d_model=cfg["d"], n_head=cfg["H"], n_layer=cfg["NL"], total_seq_length=cfg["L"],
        **({} if dropout is None else {"dropout": dropout}))
    task = tr.NextItemPredictionTask(weight_tying=True, sampled_softmax=bool(cfg.get("sampled")),
                                     max_n_samples=cfg.get("sampled") or 100)
    model = tcfg.to_torch_model(inputs, task)
    return model.to(device).eval()


def build_oracle(cfg):
    import t4r_oracle as O

    torch.manual_seed(1)
    cards = cardinalities(cfg)
    return O.OracleSessionModel(cardinalities=cards, embedding_dims={n: cfg["De"] for n in cards},
                                item_id="item_id/list", continuous=(), d_model=cfg["d"], n_head=cfg["H"],
                                n_layer=cfg["NL"], max_seq_len=cfg["L"], arch=cfg["arch"], masking=cfg["masking"],
                                sampled_softmax=bool(cfg.get("sampled")),
                                max_n_samples=cfg.get("sampled") or 100).eval()


def _oracle_step_seconds(oracle, cfg, B_cpu, steps, warmup):
    batch = synth_batch(B_cpu, cfg["L"], cfg, seed=0)
    g = torch.Generator().manual_seed(2)
    u = torch.rand((B_cpu, cfg["L"] + 2), generator=g)
    draws = {"u_bern": u[:, :cfg["L"]], "u_force": u[:, cfg["L"]], "u_unmask": u[:, cfg["L"] + 1]}
    ts = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            kw = {}
            if getattr(oracle, "sampled_softmax", False):
                # the reference draws its negatives inside the forward (model/prediction_task.py:843-845): timed
                import t4r_oracle as O
                raw = torch.multinomial(oracle.dist, 2 * oracle.max_n_samples, replacement=True)
                kw["neg_samples"] = O.negatives_from_draws(raw, oracle.max_n_samples)
            out = oracle(batch, training=True, draws=draws, **kw)
            float(out["loss"])
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
    ts.sort()
    return ts[len(ts) // 2]


def time_oracle_cpu(cfg, B_cpu, steps, warmup, budget_s=8.0):
    """The reference's CPU torch path on a bounded sample of the workload.

    The arm is given its best shot within the time bound: (1) the intra-op thread count is calibrated on one
    small step per candidate (all host threads, half, 32, 16 -- torch's CPU path re-faults its freshly
    allocated [T, V] logits every step, which gets slower, not faster, with very many threads), and (2) the
    sample grows from B_cpu sessions per step towards ~budget_s seconds per step (at most 8 x B_cpu), because
    the one pass over the item table per step is amortised over the sessions of the step exactly as in the
    full-size batch.  Returns (sessions/s, median s/step, threads used, sessions per step).
    """
    ncpu = os.cpu_count() or 1
    oracle = build_oracle(cfg)
    best_t, best_threads = None, ncpu
    for threads in sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32), min(ncpu, 16)}, reverse=True):
        torch.set_num_threads(threads)
        t = _oracle_step_seconds(oracle, cfg, B_cpu, 1, 1 if best_t is None else 0)
        if best_t is None or t < best_t:
            best_t, best_threads = t, threads
    torch.set_num_threads(best_threads)
    grow = int(max(1, min(8, budget_s // max(best_t, 1e-3))))
    # memory bound: the reference materialises [T, V] fp32 logits (plus ~3 same-sized temporaries in CrossEntropyLoss);
    # keep that under a quarter of the host memory that is free right now
    try:
        import psutil
        free = psutil.virtual_memory().available
    except Exception:
        free = 16 << 30
    labels_per_session = cfg["L"] if cfg["masking"] == "clm" else max(3.0, 0.15 * cfg["L"] + 1)
    width = (cfg.get("sampled") or cfg["V"])
    per_session = labels_per_session * width * 4 * 4
    grow = int(max(1, min(grow, (0.25 * free) // max(per_session * B_cpu, 1))))
    B_run = B_cpu * grow
    med = _oracle_step_seconds(oracle, cfg, B_run, steps, warmup)
    return B_run / med, med, best_threads, B_run


def recall_agreement(cfg, model, batch_dev, batch_host, n_sample=64):
    """BASELINE.json's accuracy anchor: Recall@20 of the evaluation forward (`testing=True`: the last item of every
    session is the label, full scores over V).  Ours = the fused head's label ranks on the whole bench batch; the
    oracle (reference CPU path, THE SAME weights copied over) scores the first `n_sample` sessions, and the label
    ranks of those sessions are compared one by one (with random-init weights Recall@20 itself is ~20/V for both,
    so the rank agreement is the informative part).  Best effort: never fails the bench line."""
    with torch.no_grad():
        out = model(batch_dev, training=False, testing=True)
        T = int(out.count.item()) if out.count is not None else int(out.row_rank.numel())
        ranks = out.row_rank[:T].long().cpu()
        oracle = oracle_with_model_weights(cfg, model)
        small = {k: v[:n_sample] for k, v in batch_host.items()}
        ref_rank = oracle_label_ranks(oracle, small)
        n = ref_rank.numel()
        mine = ranks[:n]
        return {"k": 20, "ours_full_batch": float((ranks < 20).float().mean()), "label_rows": T,
                "ours_sample": float((mine < 20).float().mean()), "oracle_sample": float((ref_rank < 20).float().mean()),
                "sample": f"first {n_sample} sessions, eval mode, oracle with the product's weights",
                "label_rank_max_abs_diff": int((mine - ref_rank).abs().max()),
                "label_rank_median_rel_diff": float(((mine - ref_rank).abs().float() / ref_rank.clamp(min=1).float()).median())}


def skewed_stream(B, L, V, seed):
    """Synthetic sessions with something to learn: log-uniform (popularity-skewed) start item -- the distribution
    LogUniformSampler assumes, model/prediction_task.py:719 -- followed by consecutive item ids; length U{2..L}."""
    import math
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(2, L + 1, (B,), generator=g)
    u = torch.rand(B, generator=g)
    start = torch.exp(u * math.log(float(V - L - 1))).long().clamp(1, V - L - 1)
    ids = start[:, None] + torch.arange(L)[None]
    return {"item_id/list": torch.where(torch.arange(L)[None] < lens[:, None], ids, torch.zeros_like(ids))}


def trained_recall(dev, steps=150, batch=512, n_eval=256):
    """A Recall@20 that is not vacuous: the config-1-size model (10K items, XLNet d=64 x2, item feature only) is
    TRAINED here, on the device, with the fused training step + FusedAdamW (SURVEY 8f N3) for `steps` steps on
    `skewed_stream`, then evaluated (`testing=True`: last item of each held-out session) by the product's fused head
    AND by the oracle -- the reference CPU path carrying the trained weights.  Reports both Recall@20 values, their
    difference, and the label-rank agreement.  (At 1M items a few hundred steps would not move Recall@20 off 0.)"""
    from transformers4rec_b200.training import FusedAdamW, FusedTrainingStep, training_loss
    cfg = dict(CONFIGS["config1"])
    B, L, V = batch, cfg["L"], cfg["V"]
    model = build_product_model(cfg, dev, dropout=0.0)
    step = FusedTrainingStep(model)
    opt = FusedAdamW(model.parameters(), lr=1e-2, weight_decay=0.0)
    first = last = None
    t0 = time.perf_counter()
    for i in range(steps):
        b = {k: v.to(dev) for k, v in skewed_stream(B, L, V, 100 + i).items()}
        opt.zero_grad(set_to_none=True)
        loss = training_loss(model, b, step)
        loss.backward()
        opt.step()
        if i == 0:
            first = float(loss.detach())
    last = float(loss.detach())
    train_s = time.perf_counter() - t0
    held = skewed_stream(n_eval, L, V, 9999)
    with torch.no_grad():
        out = model({k: v.to(dev) for k, v in held.items()}, training=False, testing=True)
        T = int(out.count.item()) if out.count is not None else int(out.row_rank.numel())
        ranks = out.row_rank[:T].long().cpu()
        oracle = oracle_with_model_weights(cfg, model)
        ref_rank = oracle_label_ranks(oracle, held)
        ref_loss = float(oracle(held, training=False, testing=True)["loss"])
    ours, ref = float((ranks < 20).float().mean()), float((ref_rank < 20).float().mean())
    return {"k": 20, "ours": ours, "oracle": ref, "abs_diff": abs(ours - ref), "eval_sessions": n_eval,
            "eval_loss_ours": float(out["loss"]), "eval_loss_oracle": ref_loss,
            "label_rank_max_abs_diff": int((ranks - ref_rank).abs().max()),
            "label_ranks_identical": float((ranks == ref_rank).float().mean()),
            "trained": f"{steps} steps x {B} sessions of FusedTrainingStep + FusedAdamW(lr 1e-2) on the device, "
                       f"{train_s:.1f} s; training loss {first:.3f} -> {last:.3f}",
            "model": "BASELINE config-1 size: 10K items, XLNet d=64 x2, item-id feature, dropout 0",
            "data": "synthetic log-uniform start item + consecutive ids (skewed_stream)",
            "note": "reference notebook anchor on real yoochoose data: Recall@20 0.505; not comparable to synthetic data"}


def oracle_label_ranks(oracle, batch):
    """Rank of every evaluation label among the oracle's full scores (ties towards the lower id, the label excluded)."""
    with torch.no_grad():
        ref = oracle(batch, training=False, testing=True)
    pred, y = ref["predictions"], ref["labels"]
    tgt = pred.gather(1, y.unsqueeze(1))
    ids = torch.arange(pred.shape[1]).unsqueeze(0)
    return (((pred > tgt) | ((pred == tgt) & (ids < y.unsqueeze(1)))) & (ids != y.unsqueeze(1))).sum(1)


def oracle_with_model_weights(cfg, model):
    """The oracle graph of `cfg` carrying the product model's parameters (device -> host copies)."""
    with torch.no_grad():
        oracle = build_oracle(cfg)
        head = model.heads[0]
        inputs, tblock = head.body[0], head.body[1]
        for name in oracle.table_names:
            oracle.tables[name.replace("/", "__")].weight.copy_(inputs.categorical_module.embedding_tables[name].weight.cpu())
        lin = inputs.projection_module[0][0]
        oracle.proj.weight.copy_(lin.weight.cpu()); oracle.proj.bias.copy_(lin.bias.cpu())
        oracle.masked_item_embedding.copy_(inputs.masking.masked_item_embedding.cpu())
        oracle.transformer.load_state_dict({k: v.cpu() for k, v in tblock.transformer.state_dict().items()}, strict=False)
        task = head.prediction_task_dict["next-item"]
        if oracle.task_block is not None:
            tl = task.task_block[0][0]
            oracle.task_block.weight.copy_(tl.weight.cpu()); oracle.task_block.bias.copy_(tl.bias.cpu())
    return oracle


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config2", choices=sorted(CONFIGS))
    ap.add_argument("--cpu-sessions", type=int, default=64, help="sessions per CPU-baseline step (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--nprod", type=int, default=2,
                    help="arithmetic of the training full-softmax head: 2 (the library default) = fp16 x fp16 + two e4m3 "
                         "cross terms (2 tensor units per MAC; device-side error table: profiles/r2_head_precision.json), "
                         "3 = split-bf16 x3, 1 = plain bf16")
    ap.add_argument("--graph", action="store_true", help="also time the step replayed from a CUDA graph")
    ap.add_argument("--no-sharded", action="store_true",
                    help="skip the `sharded` record (row-sharded configs 4 and 5 timed at this N after the headline)")
    ap.add_argument("--sharded-timeout", type=float, default=240.0,
                    help="seconds the sharded legs may take before the headline line is printed without them")
    ap.add_argument("--train", action="store_true",
                    help="time a TRAINING step instead (forward + backward through transformers4rec_b200.training + one "
                         "optimizer step); not BASELINE.json's metric -- the line says so in `metric`")
    ap.add_argument("--optimizer", choices=["sgd", "adamw"], default="sgd",
                    help="with --train: torch.optim.SGD, or FusedAdamW (the t4r_train_adamw kernel)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, under 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = dict(CONFIGS[args.workload])
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    config_desc = {"workload": f"BASELINE.json {args.workload}: {cfg['label']}", "per_gpu_batch": cfg["B"],
                   "global_batch": cfg["B"] * world, "seq_len": cfg["L"], "items": cfg["V"],
                   "parallelism": (f"item table + tied head row-sharded over {world} ranks (1 all-to-all + 1 all-gather per "
                                   f"step), everything else data parallel") if cfg.get("sharded") else
                   f"{world} independent replicas (sessions are independent; no data-path collective)",
                   "l2_policy": (f"inputs larger than L2 ({cfg['V'] * cfg['De'] * 4 / 1e9:.2f} GB item table + as much again in "
                                 f"split planes; the full-softmax head streams the planes once per step)")
                   if cfg["V"] * cfg["De"] * 8 > 126e6 else
                   "working set fits the 126 MB L2 and is not flushed (parity-test case, not the bench line)",
                   "product_arithmetic": {3: "split-bf16 x3 tcgen05 products, fp32 accumulate",
                                          2: "head: fp16 x fp16 + 2 e4m3 cross-term tcgen05 products (2 units per MAC), "
                                             "rest: split-bf16 x3; fp32 accumulate",
                                          1: "bf16 tcgen05, fp32 accumulate"}[args.nprod]}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        steps = args.steps
        warm = 1
        v, med, threads, b_run = time_oracle_cpu(cfg, args.cpu_sessions, steps, warm)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "sessions/s", "n_gpus": args.gpus,
                "steps": steps, "warmup": warm, "ms_per_step": med * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_desc,
                "cpu_baseline": {"value": v, "unit": "sessions/s", "cores": threads, "kind": "port",
                                 "sample": f"{b_run} sessions/step of the same workload, {steps} timed steps (median), "
                                           f"oracle graph = torch CPU ops + HF encoder, {threads} of "
                                           f"{os.cpu_count()} host threads (best of a calibration sweep)"},
                "e2e": {"value": v, "unit": "sessions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ product arm (B200)
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the product path has no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    want_sharded_record = (args.workload == "config2" and not args.train and not args.no_sharded)
    if world > 1 or cfg.get("sharded") or want_sharded_record:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        dist.init_process_group("nccl", device_id=dev, rank=rank, world_size=world)
    peaks, peak_kind = load_peaks()

    def emit(line):
        print(json.dumps(line), flush=True)

    res = run_workload(args, cfg, dev, rank, world, local_rank, config_desc, peaks, peak_kind, headline=True)
    line = res["line"] if rank == 0 else None
    if want_sharded_record:
        # SURVEY 8e / VERDICT r1 item 1: the row-sharded table + tied head, timed at this N next to the headline.
        # The headline above is already measured; whatever happens below (an exception, a hang) it is still printed.
        done = threading.Event()

        def watchdog():
            if done.wait(args.sharded_timeout):
                return
            if rank == 0:
                line["sharded"] = {"error": f"the sharded legs did not finish within {args.sharded_timeout} s"}
                emit(line)
            os._exit(0)
        threading.Thread(target=watchdog, daemon=True).start()
        rec = {}
        for name in ("config4", "config5"):
            try:
                rec[name] = run_sharded_leg(args, name, dev, rank, world, peaks)
            except Exception as exc:  # noqa: BLE001 -- recorded in the line; the headline stands on its own
                rec[name] = {"error": f"{type(exc).__name__}: {exc}"[:400]}
                break  # a CUDA error is sticky: do not try the next leg on a broken context
        done.set()
        if rank == 0:
            line["sharded"] = rec
    if rank == 0:
        emit(line)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        try:
            torch.distributed.destroy_process_group()
        except Exception:  # noqa: BLE001
            pass


N_ROTATE = 8   # distinct batches cycled through the timed loops: no step re-reads the table rows of the one before


def _stage_times(model, batches, K):
    """CUDA-event times (ms, mean over K steps) of the three stages of the forward on the current stream."""
    head = model.heads[0]
    inputs, tblock = head.body[0], head.body[1]
    task = head.prediction_task_dict["next-item"]
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
    with torch.no_grad():
        for i in range(K):
            b = batches[i % len(batches)]
            ev[i][0].record()
            x = inputs(b, training=True)
            ev[i][1].record()
            h = tblock(x)
            ev[i][2].record()
            task(h, training=True)
            ev[i][3].record()
    torch.cuda.synchronize()
    return [sum(e[j].elapsed_time(e[j + 1]) for e in ev) / K for j in range(3)]


def _gather_time(model, cfg, batches, K):
    """The embedding gather (K1) alone, as the model calls it, over rotating id sets (rows not L2-resident)."""
    from transformers4rec_b200 import ops
    cm = model.heads[0].body[0].categorical_module
    names = sorted(cardinalities(cfg))
    C = sum(cm.embedding_tables[n].weight.shape[1] for n in names)
    M = batches[0][names[0]].numel()

    def call(b):
        cats, col = [], 0
        for n in names:
            w = cm.embedding_tables[n].weight.detach()
            cats.append((w, b[n].reshape(-1), col))
            col += w.shape[1]
        return ops.embed_concat(cats, [], M, C, want_f32=False, want_planes=True)
    for i in range(3):
        call(batches[i % len(batches)])
    torch.cuda.synchronize()
    # the kernel runs ~20 us, less than the host needs to marshal one launch: the N_ROTATE launches are captured into a
    # CUDA graph once and replayed, so the events time the device, not the Python call overhead
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        keep = [call(b) for b in batches]
    reps = max(1, K // len(batches))
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / (reps * len(batches))
    del keep, graph
    F = len(names)
    # SURVEY 8d: gather_bytes = B*L*(8F + 4*sum(De)) read + the planes written (2 x bf16 x round_up64(C) = ~4C)
    nbytes = M * (8 * F + 4 * C) + M * 4 * ((C + 63) // 64 * 64)
    return ms, nbytes


DUMP_PREDICTION_BYTES = 48 << 20   # the sampled prediction rows; with loss and labels the dump stays under 64 MB


def dump_outputs(path, loss, task, train_step=None, seed=0):
    """Write what a caller of the timed step received from its last call as ``path/<name>.npy``: ``loss``, ``labels``
    (the targets of the masked positions, in row order) and, where the path materialises them, ``predictions`` -- the
    rows of the [T, V] scores (or [T, 1 + S] with sampled softmax) at a fixed seeded sample of label rows, whose
    indices are ``prediction_rows``; the whole matrix does not fit.  Floats are stored as float32, integers as
    float64, which holds them exactly."""
    import numpy as np

    if train_step is not None:
        arrays = {"loss": loss, "labels": train_step.labels[:train_step.T]}
    else:
        arrays = {"loss": loss, "labels": task._lazy_labels()}
        if "xt_planes" in task._last:   # over a row-sharded table the path does not materialise predictions
            arrays.update(_prediction_rows(task, seed))
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().cpu()
        np.save(os.path.join(path, f"{name}.npy"), t.numpy().astype(np.float32 if t.is_floating_point() else np.float64))


def _prediction_rows(task, seed):
    """``predictions`` of the task's last forward at a seeded sample of its label rows: the task's own materialisation
    pointed at a copy of those rows (zero-padded to whole 128-row tiles), so the scores are computed as for all rows."""
    st = task._last
    T = int(st["count"].item())
    cols = 1 + st["neg"].numel() if st["sampled"] else task.output_weight().shape[0]
    R = min(T, max(1, DUMP_PREDICTION_BYTES // (4 * cols)))
    rows = torch.randperm(T, generator=torch.Generator().manual_seed(seed))[:R].sort().values
    idx = rows.to(st["labels"].device)
    planes = st["xt_planes"]
    sub_planes = torch.zeros((planes.shape[0], (R + 127) // 128 * 128, planes.shape[2]), dtype=planes.dtype,
                             device=planes.device)
    sub_planes[:, :R] = planes[:, idx]
    sub = dict(st, xt_planes=sub_planes, labels=st["labels"][idx],
               count=torch.full((1,), R, dtype=torch.int32, device=idx.device))
    if st["sampled"]:
        sub["pos"] = st["pos"][idx]
    task._last = sub
    try:
        predictions = task._lazy_predictions()
    finally:
        task._last = st
    return {"predictions": predictions, "prediction_rows": rows}


def run_workload(args, cfg, dev, rank, world, local_rank, config_desc, peaks, peak_kind, headline):
    import transformers4rec_b200 as t4r
    from transformers4rec_b200 import ops

    lib = t4r.load()
    model = build_product_model(cfg, dev)
    task = model.heads[0].prediction_task_dict["next-item"]
    task.nprod = args.nprod
    B, L, V = cfg["B"], cfg["L"], cfg["V"]
    hosts = [{k: v.pin_memory() for k, v in synth_batch(B, L, cfg, seed=1000 * rank + j).items()} for j in range(N_ROTATE)]
    devs = [{k: v.to(dev) for k, v in h.items()} for h in hosts]
    batch_host, batch_dev = hosts[0], devs[0]
    h2d_bytes = int(sum(v.numel() * v.element_size() for v in batch_host.values()))

    def to_device(j):
        return {k: v.to(dev, non_blocking=True) for k, v in hosts[j % N_ROTATE].items()}

    train_step = opt = None
    if args.train:
        from transformers4rec_b200.training import FusedAdamW, FusedTrainingStep, training_loss
        train_step = FusedTrainingStep(model)
        opt = (FusedAdamW(model.parameters(), lr=1e-3) if args.optimizer == "adamw"
               else torch.optim.SGD(model.parameters(), lr=1e-3))

    def step(batch):
        if train_step is not None:
            opt.zero_grad(set_to_none=True)
            loss = training_loss(model, batch, train_step)
            loss.backward()
            opt.step()
            return loss.detach()
        with torch.no_grad():
            return model(batch, training=True)["loss"]

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # started before warm-up so samples exist even for a short timed region
    W = max(args.warmup, 3)
    for i in range(W):
        step(devs[i % N_ROTATE])
    barrier()

    # --- timed region 1: inputs resident in HBM, N_ROTATE distinct batches cycled
    K = args.steps
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for a, b in evs:  # torch creates the cudaEvent_t lazily: record once so .cuda_event is a live handle
        a.record(); b.record()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if rank == 0:
        sampler.lines.clear()  # keep only samples taken during the timed region (load already applied)
    n0 = lib.t4r_launch_count()
    barrier()
    e0.record()
    for i in range(K):
        ops.HEAD_EVENTS = evs[i]
        loss_last = step(devs[i % N_ROTATE])
    e1.record()
    barrier()
    ops.HEAD_EVENTS = None
    n1 = lib.t4r_launch_count()
    clocks = sampler.stop() if rank == 0 else None
    ms_total = e0.elapsed_time(e1)
    head_ms = sorted(a.elapsed_time(b) for a, b in evs)
    head_ms_avg = sum(head_ms) / len(head_ms)
    T = train_step.T if train_step is not None else int(task._last["count"].item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss_last, task, train_step)  # before any later forward replaces task._last

    # --- optional: the same step captured once and replayed from a CUDA graph (no host work at all)
    graph_ms = None
    if args.graph and not args.train:
        try:
            gph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gph):
                step(batch_dev)
            for _ in range(3):
                gph.replay()
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(K):
                gph.replay()
            g1.record()
            barrier()
            graph_ms = g0.elapsed_time(g1) / K
        except Exception as exc:  # capture is best-effort; the eager number above stands on its own
            graph_ms = f"capture failed: {type(exc).__name__}: {exc}"[:200]

    # --- timed region 2: end to end through the public API with HOST inputs
    loss_host = 0.0
    for j in range(2):
        loss_host = step(to_device(j)).item()
    barrier()
    t0 = time.perf_counter()
    for j in range(K):
        loss_host = step(to_device(j)).item()  # H2D + D2H every step
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    # the same loop with the result read ONE STEP LATE (pinned buffer + event): every step still copies its inputs H2D
    # and has its loss read on the host, but the host no longer stalls the launch of step i+1 on the loss of step i
    e2e_pipe_s = None
    if not args.train:
        try:
            bufs = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
            evs2 = [torch.cuda.Event(), torch.cuda.Event()]
            barrier()
            t0 = time.perf_counter()
            prev = None
            for j in range(K):
                loss_dev = step(to_device(j))
                bufs[j & 1].copy_(loss_dev.reshape(1), non_blocking=True)
                evs2[j & 1].record()
                if prev is not None:
                    evs2[prev].synchronize()
                    loss_host = float(bufs[prev])
                prev = j & 1
            evs2[prev].synchronize()
            loss_host = float(bufs[prev])
            torch.cuda.synchronize()
            e2e_pipe_s = time.perf_counter() - t0
        except Exception:  # noqa: BLE001 -- an extra, never at the cost of the line
            e2e_pipe_s = None

    # --- stage breakdown and the gather alone (CUDA events, rank 0's own stream; not part of `value`)
    stages = gather = None
    if not args.train and not cfg.get("sharded"):
        try:
            stages = _stage_times(model, devs, K)
            gather = _gather_time(model, cfg, devs, max(K, 20))
        except Exception as exc:  # noqa: BLE001 -- explanatory numbers never cost the line
            stages = gather = None
            print(f"[bench] stage breakdown skipped: {type(exc).__name__}: {exc}", file=sys.stderr)

    tt = torch.tensor([ms_total, e2e_s * 1e3, (e2e_pipe_s or 0.0) * 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, e2e_pipe_ms = float(tt[0]), float(tt[1]), float(tt[2])
    if rank != 0:
        del model
        torch.cuda.empty_cache()
        return {"line": None}

    ms_per_step = ms_total / K
    value = B * world / (ms_per_step / 1e3)
    e2e_value = B * world / (e2e_ms / K / 1e3)
    head_flops = 2.0 * T * V * cfg["De"]  # algorithmic (SURVEY §8d: head_flop = 2*T*V*De)
    if cfg.get("sharded"):  # per launch: the label rows of ALL ranks against this rank's V/world table rows
        head_flops = 2.0 * (T * world) * (V / world) * cfg["De"]
    if cfg.get("sampled"):  # SURVEY §8d: 2*T*(S+1)*De with S = the negatives that survived unique()[:S]
        head_flops = 2.0 * T * (int(task._last["neg"].numel()) + 1) * cfg["De"]
    achieved_tf = head_flops / (head_ms_avg * 1e-3) / 1e12
    peak_tf = float(peaks.get("bf16_tflops", peaks.get("bf16_tflops_sustained")))
    resident = os.environ.get("T4R_HEAD_RESIDENT", "1") != "0" and cfg["De"] <= 256 and not cfg.get("sampled")
    head_kernel = ("head_resident_kernel (CTA-pair tcgen05 GEMM, A tile resident in shared memory: tied logits + "
                   "online LSE)" if resident else
                   "gemm2_bf16x3_kernel<256,false,true> (CTA-pair tcgen05 GEMM: tied logits + online LSE)")
    roofline = {"bound": "tensor", "kernel": head_kernel,
                "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                "peak_source": f"{peak_kind} MEASURED_PEAKS.json bf16_tflops (burst: the timed region is a fraction of a "
                               f"second; sustained {peaks.get('bf16_tflops_sustained')} would give "
                               f"{achieved_tf / float(peaks.get('bf16_tflops_sustained', peak_tf)):.3f})",
                "traffic": head_traffic(resident) if args.workload == "config2" else None, "launch_ms": head_ms_avg,
                "share_of_step": head_ms_avg / ms_per_step,
                "algorithmic_flops_per_launch": head_flops, "label_rows_T": T,
                "note": {3: "split-bf16 x3 issues 3 tensor-core MACs per algorithmic MAC: frac <= 1/3 by construction",
                         2: "fp16 + 2 x e4m3 cross terms: 2 bf16-equivalent tensor passes per MAC: frac <= 1/2",
                         1: "plain bf16 product"}[args.nprod]}
    line = {"metric": METRIC if not args.train else "sessions/sec (fwd+bwd+%s step; NOT the BASELINE metric)" % args.optimizer, "value": value, "unit": "sessions/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {3: "f32 (bf16 hi/lo split operands on tcgen05, fp32 accumulate)",
                                           2: "f32 (head: fp16 + e4m3 cross terms on tcgen05; rest bf16 hi/lo split)",
                                           1: "bf16"}[args.nprod], "data": "synthetic", "config": config_desc, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "sessions/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 4, "loss": loss_host,
                    "how": "model(batch)['loss'].item() every step: pinned-host ids copied H2D, the loss read back before "
                           "the next step is launched",
                    "pipelined_value": (B * world / (e2e_pipe_ms / K / 1e3)) if e2e_pipe_ms > 0 else None,
                    "pipelined_how": "same copies and reads, the loss of step i read after step i+1 has been launched"},
            "gpu_launches": int(n1 - n0), "roofline": roofline}
    if stages is not None:
        enc_flops = cfg["NL"] * B * L * (24 * cfg["d"] ** 2 + 8 * L * cfg["d"])      # SURVEY §8d enc_flop
        enc_tf = enc_flops / (stages[1] * 1e-3) / 1e12
        line["stages_ms"] = {"input_block": stages[0], "encoder": stages[1], "head": stages[2],
                             "how": "CUDA events between the three module calls, mean over the timed steps, separate pass"}
        line["roofline_encoder"] = {"bound": "tensor", "achieved": enc_tf, "peak": peak_tf, "unit": "TFLOP/s",
                                    "frac": enc_tf / peak_tf, "ms": stages[1], "algorithmic_flops": enc_flops,
                                    "note": "whole encoder (QKV, relative attention, O-proj + LN, fused FFN; 3 tensor "
                                            "passes per MAC in the GEMMs)",
                                    "ncu_tensor_pipe": ncu_tensor_pipe()}
    if gather is not None:
        g_ms, g_bytes = gather
        hbm = float(peaks.get("hbm_gbs", 6482.4))
        line["roofline_gather"] = {"bound": "hbm", "kernel": "embed_concat_kernel", "achieved": g_bytes / (g_ms * 1e-3) / 1e9,
                                   "peak": hbm, "unit": "GB/s", "frac": g_bytes / (g_ms * 1e-3) / 1e9 / hbm,
                                   "launch_ms": g_ms, "algorithmic_bytes_per_launch": g_bytes,
                                   "how": f"{N_ROTATE} distinct id sets cycled (table rows not L2-resident), the launches "
                                          f"replayed from a CUDA graph, CUDA events around the replays"}
    if graph_ms is not None:
        line["cuda_graph"] = {"ms_per_step": graph_ms, "value": (B * world / (graph_ms / 1e3)) if isinstance(graph_ms, float) else None}
    if not args.no_cpu_baseline and world == 1:
        v, med, threads, b_run = time_oracle_cpu(cfg, args.cpu_sessions, 3, 1)
        line["cpu_baseline"] = {"value": v, "unit": "sessions/s", "cores": threads, "kind": "port",
                                "sample": f"{b_run} sessions/step of the same workload, 3 timed steps "
                                          f"(median {med:.2f} s), oracle graph = torch CPU ops + HF encoder, {threads} of "
                                          f"{os.cpu_count()} host threads (best of a calibration sweep)"}
    if not args.no_cpu_baseline and world == 1 and not cfg.get("sharded") and not args.train:
        try:
            line["recall_at_20"] = recall_agreement(cfg, model, batch_dev, batch_host)
        except Exception as exc:  # an accuracy side-note must never cost the throughput line
            line["recall_at_20"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        try:
            line["recall_at_20_trained"] = trained_recall(dev)
        except Exception as exc:  # noqa: BLE001
            line["recall_at_20_trained"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    del model
    torch.cuda.empty_cache()
    return {"line": line}


SHARDED_LEGS = {
    # BASELINE.json configs[3]: 10M-row table, block-sharded over the N ranks (N = 1: the whole table on one GPU),
    # tied full-softmax head, B = 2048 per GPU.  Per-rank head work T_global * V / N is constant in N: weak scaling.
    "config4": dict(V=10_000_001, De=256, d=256, H=8, NL=4, L=20, B=2048, arch="xlnet", masking="mlm", sharded=True),
    # BASELINE.json configs[4]: 50M-row table sharded over the N ranks, sampled softmax with 50K negatives, L = 50.
    "config5": dict(V=50_000_001, De=256, d=256, H=8, NL=4, L=50, B=2048, arch="xlnet", masking="mlm", sharded=True,
                    sampled=50_000),
}


def _time_loop(fn, K, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / K


def run_sharded_leg(args, name, dev, rank, world, peaks):
    """One row-sharded workload at this N: whole-step sessions/s (max over ranks) plus the pieces that move data
    between GPUs, each timed alone with CUDA events: the peer-memory lookup, the label-row pull, the two 4-byte
    ordering collectives -- and the head GEMM's own time from its event pair."""
    import torch.distributed as dist

    from transformers4rec_b200 import distributed as D
    from transformers4rec_b200 import ops
    cfg = dict(SHARDED_LEGS[name])
    B, L, V, De = cfg["B"], cfg["L"], cfg["V"], cfg["De"]
    model = build_product_model(cfg, dev)
    task = model.heads[0].prediction_task_dict["next-item"]
    task.nprod = args.nprod
    inputs = model.heads[0].body[0]
    table = inputs.categorical_module.embedding_tables["item_id/list"]
    devs = [{k: v.to(dev) for k, v in synth_batch(B, L, cfg, seed=1000 * rank + j).items()} for j in range(N_ROTATE)]

    def step(i):
        with torch.no_grad():
            return model(devs[i % N_ROTATE], training=True)["loss"]
    K = args.steps
    for i in range(3):
        step(i)
    dist.barrier(); torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for a, b in evs:
        a.record(); b.record()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier(); torch.cuda.synchronize()
    e0.record()
    loss = None
    for i in range(K):
        ops.HEAD_EVENTS = evs[i]
        loss = step(i)
    e1.record()
    dist.barrier(); torch.cuda.synchronize()
    ops.HEAD_EVENTS = None
    ms = e0.elapsed_time(e1) / K
    head_ms = sum(a.elapsed_time(b) for a, b in evs) / K
    T = int(task._last["count"].item())
    peer = table.peer_view() is not None
    rec = {"exchange": "nvlink peer memory (t4r_peer_* kernels)" if peer else "nccl all-gather + all-to-all"}
    # pieces, each alone
    n_ids = B * L
    ids_flat = devs[0]["item_id/list"].reshape(-1)
    lookup_ms = _time_loop(lambda: table.lookup(ids_flat), 10)
    rec["lookup"] = {"ms": lookup_ms, "rows": n_ids, "bytes": n_ids * De * 4,
                     "remote_bytes": int(n_ids * De * 4 * (world - 1) / world * 0.55),
                     "note": "item rows of one batch from their owners' shards; ~45 % of the positions are the padding id, "
                             "served from a per-CTA copy of that row (remote_bytes counts the other 55 % x (N-1)/N)"}
    if cfg.get("sampled"):
        S = int(task._last["S"])
        neg = torch.randint(1, V, (S,), device=dev)
        neg_ms = _time_loop(lambda: table.lookup(neg), 10)
        rec["negatives_lookup"] = {"ms": neg_ms, "rows": S, "bytes": S * De * 4,
                                   "remote_bytes": int(S * De * 4 * (world - 1) / world)}
        head_flops = 2.0 * T * (S + 1) * De
        colls = ["broadcast of the raw negative draws (2 x 50 000 int64)", "all-reduce of (sum of row losses, T)"]
    else:
        ph = getattr(task, "_peer_head_state", None)
        if peer and ph is not None and ph.ok:
            cnt = task._last["count"]
            pull_ms = _time_loop(lambda: ops.peer_pull_rows(ph.views[0], ph.views[1], ph.counts, ph.cap, De), 10)
            bar_ms = _time_loop(lambda: (dist.all_gather_into_tensor(ph.counts, cnt.reshape(1).to(torch.int32), group=ph.group),
                                         dist.all_reduce(ph.token, group=ph.group)), 10)
            t_tot = int(ph.counts.sum().item())
            rec["label_row_pull"] = {"ms": pull_ms, "rows": t_tot, "bytes": t_tot * De * 4,
                                     "remote_bytes": int((t_tot - T) * De * 4)}
            rec["stats_exchange"] = {"bytes": t_tot * 12 * max(world - 1, 0),
                                     "note": "peer_combine_lse reads 12 B per row from every other shard; its time is "
                                             "inside ms_per_step"}
            rec["ordering_collectives"] = {"ms": bar_ms, "bytes": 8,
                                           "what": "4-byte all-gather of the label-row counts + 4-byte all-reduce"}
            colls = ["all-gather of counts (4 B)", "all-reduce token (4 B)"]
        else:
            colls = ["all-gather of ids", "all-to-all of rows", "all-gather of counts", "all-gather of label rows",
                     "all-gather of labels", "all-gather of (lse, label logit)"]
        head_flops = 2.0 * (T * world) * (V / world) * De
    tt = torch.tensor([ms], device=dev, dtype=torch.float64)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms = float(tt[0])
    value = B * world / (ms / 1e3)
    peak_tf = float(peaks.get("bf16_tflops", 1719.6))
    rec.update({"workload": f"BASELINE.json {name}: {V:,}-row item table row-sharded over {world} rank(s), "
                            + ("sampled softmax 50 000 negatives, seq_len=50" if cfg.get("sampled") else "tied full softmax, seq_len=20")
                            + f", XLNet-base d=256 x4, MLM, batch={B} per GPU",
                "value": value, "unit": "sessions/s", "ms_per_step": ms, "steps": K, "n_gpus": world,
                "rows_per_rank": table.weight.shape[0], "label_rows_T_this_rank": T, "loss": float(loss),
                "head_gemm_ms": head_ms, "head_tflops_algorithmic": head_flops / (head_ms * 1e-3) / 1e12,
                "head_frac_of_bf16_peak": head_flops / (head_ms * 1e-3) / 1e12 / peak_tf,
                "nccl_collectives_per_step": colls, "scaling": "weak"})
    # own efficiency v_N / (N * v_1): v_1 is read from the N = 1 run of the same session when it left its note
    note = os.path.join(tempfile.gettempdir(), "t4r_bench_sharded_n1.json")
    try:
        if rank == 0 and world == 1:
            prev = {}
            if os.path.exists(note):
                with open(note) as f:
                    prev = json.load(f)
            prev[name] = value
            with open(note, "w") as f:
                json.dump(prev, f)
        if rank == 0 and world > 1 and os.path.exists(note):
            with open(note) as f:
                v1 = json.load(f).get(name)
            if v1:
                rec["efficiency_vs_n1"] = value / (world * v1)
                rec["v1"] = v1
    except Exception:  # noqa: BLE001
        pass
    del model, table, inputs, task
    torch.cuda.empty_cache()
    return rec


if __name__ == "__main__":
    main()
