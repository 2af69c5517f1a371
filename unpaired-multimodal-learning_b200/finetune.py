"""UML fine-tuning over HBM-resident feature banks - drop-in for the hot path of the reference's
``vision_language/finetune.py``.

Same entry points and argument meaning: ``train`` (:120), ``validate`` (:291), ``setup`` (:323),
``sweep`` (:406), ``main`` (:451), ``hparam_str`` (:58), ``savedir`` (:67), ``fetch_next`` (:33), the
``-c/-s/-d/-f/-o`` CLI (:513-555), the YAML sweep files, ``test_result.pth`` / ``results.pth`` outputs.

What differs, by design (SURVEY.md section 0): the reference decodes JPEGs and runs the frozen backbone
inside every step; here image AND text features come from banks written by ``features.py`` and stay in
HBM, loaders yield index batches (bit-exact sampler order), and one step is a handful of hand-written
CUDA kernels (``engine/trainer.py``) instead of an autograd graph with three backward sweeps.
Per-step diagnostics that cost a device sync each (grad cosine, CKA on re-encoded images, finetune.py
:197-244) are opt-in and evaluated at eval cadence.
"""
from __future__ import annotations

import argparse
import os
import sys
from itertools import product

import time

import torch

from . import ops
from .engine.config import parser
from .engine.datasets.utils import (BankLoader, FeatureBank, IndexBatch, TextTensorDataset,
                                    get_few_shot_setup_name, local_slice)
from .engine.models.head import (CLIP_EMBED_DIM, LANGUAGE_HIDDEN, UML, VISION_NUM_FEATURES, UMLClip, _width)
from .engine.optimizer.default import HYPER_DICT
from .engine.optimizer.optim import build_optimizer
from .engine.optimizer.scheduler import build_lr_scheduler
from .engine.tools.utils import Tee, makedirs, set_random_seed
from .engine.trainer import StepEngine
from .features import img_outdir, load_feature_bank, load_image_bank, load_text_bank, text_outdir

EVAL_FREQ = 100  # evaluate on the val bank every 100 iterations (early stopping)
FLAG = 0         # 1: run although the experiment directory already holds a result


def fetch_next(loader, loader_iter):
    """Next batch; when the epoch is exhausted build a fresh iterator (new permutation) first."""
    try:
        return next(loader_iter), loader_iter
    except StopIteration:
        loader_iter = iter(loader)
        return next(loader_iter), loader_iter


def clip_outdim(model_name):
    return _width(model_name, CLIP_EMBED_DIM, "CLIP encoder")


def vision_model_outdim(model_name):
    return _width(model_name, VISION_NUM_FEATURES, "vision model")


def language_model_outdim(model_name):
    return _width(model_name, LANGUAGE_HIDDEN, "language model")


def hparam_str(optim, lr, wd, batch_size, iters, dropout, learnable_temp):
    parts = [f"optim_{optim}", f"lr_{lr}", f"wd_{wd}", f"bs_{batch_size}", f"iters_{iters}"]
    if dropout is not None:
        parts.append(f"dropout_{dropout}")
    if learnable_temp is True:
        parts.append("learnable_temp")
    return "-".join(parts)


def savedir(outdir, dataset, encoder, train_shot, seed, text_type, text_shots, image_augmentation, mode,
            init_mode="zeroshot", alpha=0.0, text_bs=0, custom_name="", args=None):
    bench = f"{dataset}-{get_few_shot_setup_name(train_shot, seed)}"
    text_name = f"text_{text_type}" + (f"_n_{text_shots}" if text_shots is not None else "")
    image_name = f"image_{image_augmentation}_{custom_name}"
    if mode == "crossmodal":
        mod = f"finetune-{text_name}-{image_name}-alpha_{alpha}"
    elif mode == "image":
        mod = f"finetune-{image_name}"
    else:
        mod = text_name
    if text_bs > 0:
        mod += f"-text_bs_{text_bs}"
    if args is not None and mode != "crossmodal":
        mod += f"-common_dim_{args.common_dim}"
    return os.path.join(outdir, bench, encoder.replace("/", "-"), mod, init_mode)


# ------------------------------------------------------------------------------------------------
# evaluation
# ------------------------------------------------------------------------------------------------

def _dist():
    d = torch.distributed
    if d.is_available() and d.is_initialized() and d.get_world_size() > 1:
        return d.get_rank(), d.get_world_size()
    return 0, 1


def _dbg(msg):
    if os.environ.get("UML_BENCH_VERBOSE"):
        torch.cuda.synchronize()
        print(f"[train] {msg}", file=sys.stderr, flush=True)


def validate_enqueue(model, val_loader, s_img=None):
    """Launches the evaluation of ``validate`` and returns ``(loss, hits, n_rows)`` - two one-element DEVICE tensors
    and the row count - without synchronising; callers that evaluate many heads read them back together.  ``s_img``:
    the model's image temperature when the caller has already read it (a learnable one lives on the device)."""
    iter(val_loader)  # a DataLoader iterator draws a base seed from the global RNG; keep the stream aligned
    bank, bs = val_loader.bank, val_loader.batch_size
    n = len(bank)
    dev = bank.device
    s_img = float(model.scales()[0]) if s_img is None else float(s_img)
    row_loss = torch.empty(n, device=dev)
    row_pred = torch.empty(n, device=dev, dtype=torch.int32)
    W = model.head.weight.data
    adapter = model.img_proj is not None
    # The reference evaluates in fp32.  The bf16 tensor-core forward is used only where the model is trained through the
    # bf16 path as well (precision "bf16", or "auto" with a throughput-sized training batch - train() notes that on the
    # model): a run that trains on the exact path also reports fp32 accuracies and takes its early-stopping decisions on them.
    prec = getattr(model, "precision", "auto")
    want_tc = prec == "bf16" or (prec == "auto" and getattr(model, "_trained_bf16", False))
    use_tc = (want_tc and n >= 4096 and W.shape[1] % 8 == 0 and W.shape[0] <= 1024 and bank.dim % 8 == 0)
    if use_tc:
        x16 = bank.bf16()
        if adapter:  # Z = X Wp^T on the tensor cores
            z16 = torch.empty((n, W.shape[1]), device=dev, dtype=torch.bfloat16)
            ops.gemm_bf16(x16, ops.cast_bf16(model.img_proj.weight.data), z16, n, W.shape[1], bank.dim)
            x16 = z16
        segs = ops.tc_segments([n], [s_img], [1.0])
        # hit flags instead of predicted classes: the kernel needs no index tracking for them
        tws = getattr(bank, "_eval_tile_ws", None)  # scratch of the exchange forward kernel, kept with the bank
        if tws is None or tws.numel() < 16 + ((n + 255) // 256) * 264 + n * 32:
            tws = bank._eval_tile_ws = ops.tile_workspace(n, dev)
        ops.head_fwd_ce_bf16(x16, ops.cast_bf16(W), bank.labels32(), segs, None, row_loss, row_correct=row_pred, tile_ws=tws)
        hit_labels = None
    else:
        hit_labels = bank.labels
        feats = model.extract_features(bank.features) if adapter else bank.features
        ops.eval_f32(feats, bank.labels, W, s_img, row_loss, row_pred)
    out_loss = torch.empty(1, device=dev)
    out_hits = torch.empty(1, device=dev, dtype=torch.int32)
    ops.eval_reduce(row_loss, row_pred, hit_labels, bs, out_loss, out_hits)
    return out_loss, out_hits, n


def validate_group_enqueue(group, models, heads, val_loader_of):
    """``validate_enqueue`` for the running heads of a sweep group (``engine/sweep.py`` HeadGroup): heads whose
    loaders share one bank and batch size are evaluated by ONE logits + argmax launch and ONE reduction launch (the head is
    a grid dimension, the weights are read straight from the group's slab) instead of two launches per head.  Returns one
    ``(loss, hits, n_rows)`` triple per head, in the order of ``heads``; the tensors are views of per-bank result vectors
    that are read back together by the caller."""
    out = [None] * len(heads)
    by_bank = {}
    for pos, k in enumerate(heads):
        ld = val_loader_of(k)
        iter(ld)  # every DataLoader iterator draws a base seed from its generator: keep each head's stream aligned
        by_bank.setdefault((id(ld.bank), ld.batch_size), []).append((pos, k, ld))
    for (_, bs), members in by_bank.items():
        bank = members[0][2].bank
        n, dev = len(bank), bank.device
        ids = [k for _, k, _ in members]
        scales = [float(models[k].scales()[0]) for k in ids]
        row_loss = torch.empty((len(ids), n), device=dev)
        row_pred = torch.empty((len(ids), n), device=dev, dtype=torch.int32)
        ops.eval_group_f32(bank.features, bank.labels, group.W, group.W.stride(0), ids, scales, group.C, row_loss, row_pred)
        out_loss = torch.empty(len(ids), device=dev)
        out_hits = torch.empty(len(ids), device=dev, dtype=torch.int32)
        ops.eval_reduce_group(row_loss, row_pred, bank.labels, bs, out_loss, out_hits)
        for j, (pos, _, _) in enumerate(members):
            out[pos] = (out_loss[j:j + 1], out_hits[j:j + 1], n)
    return out


def alignment_probe(model, image_rows, image_labels, text_rows, n_classes, topk=10):
    """The feature probes the reference computes beside its loop when ``capture_features_during_training`` is set
    (finetune.py:209-233), on feature rows and on the device: the image rows go through ``model.extract_features`` (the
    adapter, or nothing for a CLIP head), then
      * ``cka``: linear CKA between the per-class means of those features and ``text_rows`` (one text row per class:
        ``text_rows.shape[0] == n_classes``),
      * ``mknn``: mutual 10-NN accuracy between the features and ``text_rows`` (when the two have the same number of rows),
      * ``inclass_distance``: mean over classes of the mean distance of a class's features to their mean.
    Returns a dict of floats (one read-back); a probe whose row counts do not match is left out."""
    feats = model.extract_features(image_rows.to(torch.float32)).contiguous()
    labels = image_labels.to(feats.device, torch.int64)
    counts = torch.bincount(labels, minlength=n_classes).clamp_min(1).to(feats.dtype)
    means = torch.zeros(n_classes, feats.shape[1], device=feats.device, dtype=feats.dtype).index_add_(0, labels, feats) / counts[:, None]
    dist = (feats - means[labels]).norm(dim=1)
    inclass = (torch.zeros(n_classes, device=feats.device).index_add_(0, labels, dist) / counts).mean().view(1)
    text = text_rows.to(feats.device, torch.float32).contiguous()
    parts, names = [inclass], ["inclass_distance"]
    if text.shape[0] == n_classes:
        parts.append(ops.cka_linear(means, text))
        names.append("cka")
    if text.shape[0] == feats.shape[0]:
        parts.append(ops.mutual_knn(feats, text, topk))
        names.append("mknn")
    return dict(zip(names, torch.cat(parts).tolist()))


def validate(model, val_loader, device="cuda"):
    """(val_loss, val_acc) over the loader's bank: accuracy over all rows, loss = mean over the
    loader's batches of the batch-mean CE (the reference's weighting, finetune.py:310-312).  One logit +
    argmax kernel streams the bank; logits never reach the host."""
    out_loss, out_hits, n = validate_enqueue(model, val_loader)
    return float(out_loss.item()), int(out_hits.item()) / n


# ------------------------------------------------------------------------------------------------
# training
# ------------------------------------------------------------------------------------------------

_local_slice = local_slice  # kept under its old name for callers of this module


def train(model, image_loader, text_loader, val_loader, test_loader, optimizer, scheduler, device="cuda",
          max_iters=1000, alpha=1.0, eval_freq=EVAL_FREQ, patience=5, capture_features_during_training=False,
          features_pth="./", args=None, logger=None, trace=None, stats_to_host="eval"):
    """The UML loop (reference finetune.py:120-288).  ``trace`` (optional dict) receives the host-side
    index batches and per-step stats - used by the parity tests.  ``stats_to_host``: "eval" reads the
    per-step losses back once per evaluation; "step" pushes each step's record to pinned host memory
    with an asynchronous copy (what a per-step logger needs), still without stalling the stream."""
    if stats_to_host not in ("eval", "step"):
        raise ValueError("stats_to_host must be 'eval' or 'step'")
    out = {"iter": None, "val_acc": None, "model": None, "val_classwise": None, "val_loss": None, "model_records": []}
    if trace is not None:
        trace["engine"] = None
    assert image_loader is not None or text_loader is not None, "At least one of the loaders should be provided"
    if capture_features_during_training:
        print("=> capture_features_during_training is a per-step diagnostic outside the hot path; ignored")
    model.train()
    rank, world = _dist()
    bs_i = image_loader.batch_size if image_loader is not None else 0
    bs_t = text_loader.batch_size if text_loader is not None else 0
    precision = getattr(args, "precision", None) or getattr(model, "precision", "auto")

    def per_rank(loader, bs):  # a sharded (per-rank) loader's batch size already is the local one
        return bs if (loader is not None and getattr(loader, "shard_of", None)) else -(-bs // world)

    engine = StepEngine(model, optimizer, device, per_rank(image_loader, bs_i), per_rank(text_loader, bs_t),
                        log_slots=min(max(int(eval_freq), 1), int(max_iters)) + 1, precision=precision,
                        dist_group=None, world_size=world)
    model._trained_bf16 = bool(engine._use_bf16(engine.max_rows))  # validate() follows the training path's precision
    if trace is not None:
        trace["engine"] = engine
        if trace.get("profile"):
            engine.profile = {}
    image_iter = iter(image_loader) if image_loader is not None else None
    text_iter = iter(text_loader) if text_loader is not None else None
    no_improve = 0
    pending = []  # steps whose stats have not been read back yet
    last = {"image_loss": 0.0, "text_loss": 0.0, "img_acc": 0.0, "text_acc": 0.0}

    def flush():
        nonlocal last
        if not pending:
            return
        recs = engine.read_log([s for s, _ in pending], from_host_ring=(stats_to_host == "step"))
        for (slot, lr), rec in zip(pending, recs):
            if trace is not None:
                trace.setdefault("stats", []).append(dict(rec, lr=lr))
            if logger is not None:
                logger.log({"train/image_loss": rec["image_loss"], "train/text_loss": rec["text_loss"],
                            "train/image_acc": rec["img_acc"], "train/text_acc": rec["text_acc"], "train/lr": lr})
        last = recs[-1]
        pending.clear()

    # Steps are enqueued in chunks that end at the next evaluation point, so that the host issues ONE library
    # call per chunk instead of a Python round trip per kernel; the loaders are advanced in the reference's order
    # (image batch, then text batch, per step) so the sampler stream is unchanged.
    grad_diag = bool(getattr(args, "grad_diagnostics", False) or (trace is not None and trace.get("grad_diagnostics")))
    per_step = trace is not None and bool(trace.get("record_weights"))
    # small chunks: the host prepares chunk c+1 (sampler draws, index uploads) while the GPU runs chunk c
    max_chunk = 1 if per_step else 16
    # Chunk sizes ramp up 1, 1, 2, 2, 4, 4, ... after every point where the queue is empty (start, evaluations): each
    # size is used twice so that preparing a chunk (sampler + uploads, ~0.1 ms per step) never takes longer than the
    # GPU needs for the chunk already queued (plain doubling does: the GPU then idles during the whole ramp).
    ramp = 2  # the chunk size is ramp // 2
    # trace["timing"] = {"warmup": W}: wall-clock seconds of iterations W.. (stream-synchronised on both sides,
    # including the read-back of their stats) land in trace["timing"]["seconds"] - bench.py's end-to-end arm
    timing = trace.get("timing") if trace is not None else None
    t_start = None
    i = 0
    stop = False
    while i < max_iters and not stop:
        next_eval = i if i % eval_freq == 0 else (i // eval_freq + 1) * eval_freq
        n = min(next_eval, max_iters - 1) - i + 1
        n = max(1, min(n, max_chunk, 1 << ((ramp // 2) - 1)))
        ramp = min(ramp + 1, 2 * (max_chunk.bit_length()))
        if timing is not None:
            if i < timing["warmup"]:
                n = min(n, timing["warmup"] - i)
            elif t_start is None:
                flush()
                torch.cuda.current_stream().synchronize()
                t_start = time.perf_counter()
                ramp = 3
                n = min(n, 1)
        batches, lrs = [], []
        while len(batches) < n:
            # whole runs of batches inside the current epochs are taken at once (one sampler wait and, for per-step
            # uploads, one host->device copy per loader); a step where a loader starts a new epoch goes through
            # fetch_next so that the loaders draw from the global generator in the reference's order
            k = n - len(batches)
            for it_ in (image_iter, text_iter):
                if it_ is not None:
                    k = min(k, it_.batches_left() if hasattr(it_, "batches_left") else 0)
            if k >= 1:
                imgs = image_iter.take_chunk(k) if image_iter is not None else [None] * k
                txts = text_iter.take_chunk(k) if text_iter is not None else [None] * k
            else:
                img = txt = None
                if image_iter is not None:
                    img, image_iter = fetch_next(image_loader, image_iter)
                if text_iter is not None:
                    txt, text_iter = fetch_next(text_loader, text_iter)
                imgs, txts = [img], [txt]
            for img, txt in zip(imgs, txts):
                if trace is not None and trace.get("indices", True):
                    if img is not None:
                        trace.setdefault("img_idx", []).append(img.host_idx.clone())
                    if txt is not None:
                        trace.setdefault("txt_idx", []).append(txt.host_idx.clone())
                batches.append((img, txt))
                lrs.append(scheduler.get_last_lr()[0])
                scheduler.step()
                if t_start is not None:
                    timing["rows"] = timing.get("rows", 0) + sum((b.global_n or b.n) for b in (img, txt) if b is not None)
        engine.run(batches, alpha, lrs, slot0=i)
        _dbg(f"chunk at {i} (+{n}) done")
        if stats_to_host == "step":
            engine.copy_slots_to_host(i, n)
        for j in range(n):
            pending.append((i + j, lrs[j]))
        if per_step:
            trace.setdefault("weights", []).append({k: v.detach().cpu().clone() for k, v in model.state_dict().items()})
        i += n
        last_step = i - 1

        if last_step % eval_freq == 0:
            ramp = 2
            flush()
            if grad_diag:
                # the reference's per-step gradient probes (finetune.py:190-206), here at evaluation cadence on the
                # chunk's last batches and at the weights after that step
                diag = engine.grad_diagnostics(*engine.local_batches(batches[-1]))
                if trace is not None:
                    trace.setdefault("grad_diag", []).append((last_step, diag))
                if logger is not None:
                    logger.log(dict(diag, iter=last_step))
            snapshot = {k: v.detach().clone() for k, v in model.state_dict().items()}
            _dbg("before validate")
            val_loss, val_acc = validate(model, val_loader, device=device)
            _dbg("after validate")
            testlog = ""
            if test_loader is not None:
                _, test_acc = validate(model, test_loader, device=device)
                testlog = f" | Test Acc: {test_acc:.4f}"
            if out["val_acc"] is None or val_acc > out["val_acc"]:
                out.update(iter=last_step, val_acc=val_acc, val_loss=val_loss,
                           model={k: v.cpu() for k, v in snapshot.items()})
                no_improve = 0
            else:
                no_improve += 1
            if trace is not None:
                trace.setdefault("evals", []).append((last_step, val_loss, val_acc))
            if logger is not None:
                logger.log({"val/val_loss": val_loss, "val/val_acc": val_acc, "iter": last_step})
            probe = (trace or {}).get("alignment") or getattr(args, "alignment_samples", None)
            if probe:  # {"image": (rows, labels), "text": rows}: the reference's feature probes, at evaluation cadence
                al = alignment_probe(model, probe["image"][0], probe["image"][1], probe["text"], model.head.weight.shape[0])
                if trace is not None:
                    trace.setdefault("alignment_log", []).append((last_step, al))
                if logger is not None:
                    logger.log(dict({f"train/{k}": v for k, v in al.items()}, iter=last_step))
            if rank == 0:
                print(f"Iter {last_step} | Img Loss: {last['image_loss']:.4f} | Text Loss: {last['text_loss']:.4f} | "
                      f"Img Acc: {last['img_acc']:.4f} | Text Acc: {last['text_acc']:.4f} | Val Loss: {val_loss:.4f} | "
                      f"Val Acc {val_acc:.4f}{testlog} | Count {no_improve}/{patience}")
            if no_improve >= patience:
                print(f"=> Early stopping at Iter {last_step}")
                stop = True
    flush()
    if timing is not None and t_start is not None:
        torch.cuda.current_stream().synchronize()
        timing["seconds"], timing["iters"] = time.perf_counter() - t_start, i - timing["warmup"]
    print(f"{torch.cuda.memory_allocated(0) / (1024 ** 3):.4f} GB allocated after training")
    model.load_state_dict(out["model"])
    engine.invalidate_shadow()
    val_loss, val_acc = validate(model, val_loader, device=device)
    if logger is not None:
        logger.log({"val/best_val_loss": val_loss, "val/best_val_acc": val_acc, "iter": out["iter"]})
    print(f"=> Best Val Loss {val_loss:.4f}, Val Acc {val_acc:.4f} at Iter {out['iter']}")
    return out


def train_group(models, image_loaders, text_loaders, val_loaders, test_loaders, optimizers, schedulers, device="cuda",
                max_iters=1000, alphas=1.0, eval_freq=EVAL_FREQ, patience=5, loggers=None, traces=None, tags=None):
    """K runs of ``train`` advanced in lock step over shared banks (sweep-level batching, SURVEY §8 f-1): one step of all
    K heads is two launches (``engine/sweep.py``, ``csrc/sweep.cu``) instead of K latency-bound steps.  When every head
    has an image adapter or learnable temperatures (preset ``linear``) the heads form an ``AdapterHeadGroup`` instead
    (up to five launches per step) and are evaluated head by head with ``validate_enqueue``.

    Every argument that ``train`` takes once is a list with one entry per head (``max_iters``, ``alphas`` and
    ``patience`` may be scalars); returns the list of ``train``'s result dicts.  Head k follows exactly the loop of
    ``train`` - evaluation at ``i % eval_freq == 0``, strict-improvement early stopping, best state restored - with
    its own sampler stream: its loaders draw their seeds from their own ``rng`` generator in the order a stand-alone
    run draws them from the global generator, so head k reproduces ``torch.manual_seed(s); train(...)`` when its
    generator was seeded with ``s``.  (The reference's sequential sweep lets one global stream run through all
    combinations; the order inside each run is the same, the seeds differ.)"""
    from .engine import sweep as sweep_mod

    K = len(models)
    as_list = lambda x: list(x) if isinstance(x, (list, tuple)) else [x] * K
    max_iters, alphas, patience = as_list(max_iters), [float(a) for a in as_list(alphas)], as_list(patience)
    image_loaders = as_list(image_loaders) if image_loaders is not None else [None] * K
    text_loaders = as_list(text_loaders) if text_loaders is not None else [None] * K
    test_loaders = as_list(test_loaders) if test_loaders is not None else [None] * K
    loggers = as_list(loggers) if loggers is not None else [None] * K
    traces = as_list(traces) if traces is not None else [None] * K
    tags = as_list(tags) if tags is not None else [f"head {k}" for k in range(K)]
    adapter = all(m.img_proj is not None or getattr(m, "learnable_temp", False) for m in models)
    blockers = sweep_mod.adapter_group_blockers if adapter else sweep_mod.group_blockers
    why = blockers(models, optimizers, image_loaders, text_loaders)
    if _dist()[1] > 1:
        why.append("data-parallel runs are not batched")
    if why:
        raise ValueError("train_group: " + "; ".join(why))
    has_img, has_txt = image_loaders[0] is not None, text_loaders[0] is not None
    assert has_img or has_txt, "At least one of the loaders should be provided"
    il0, tl0 = image_loaders[0], text_loaders[0]
    for m in models:
        m.train()
    log_slots = min(max(int(eval_freq), 1), int(max(max_iters))) + 1
    group = (sweep_mod.AdapterHeadGroup if adapter else sweep_mod.HeadGroup)(
        models, optimizers, il0.bank if has_img else None, tl0.bank if has_txt else None,
        il0.batch_size if has_img else 0, tl0.batch_size if has_txt else 0, device, log_slots=log_slots)
    outs = [{"iter": None, "val_acc": None, "model": None, "val_classwise": None, "val_loss": None, "model_records": []}
            for _ in range(K)]
    for tr in traces:
        if tr is not None:
            tr["engine"] = group
    # the reference's order per run: iter(image_loader), iter(text_loader) (finetune.py:157-158)
    img_it, txt_it = [None] * K, [None] * K
    for k in range(K):
        if has_img:
            img_it[k] = iter(image_loaders[k])
        if has_txt:
            txt_it[k] = iter(text_loaders[k])
    running = [max_iters[k] > 0 for k in range(K)]
    no_improve = [0] * K
    pending = []  # (step, lrs of the step) whose stats have not been read back yet
    last = None

    def flush():
        nonlocal last
        if not pending:
            return
        cols = group.read_log([s for s, _, _ in pending], has_img, has_txt)
        for j, (_, lrs, act) in enumerate(pending):
            for k in range(K):
                if not act[k] or (traces[k] is None and loggers[k] is None):
                    continue
                rec = {"image_loss": cols["image_loss"][j][k], "text_loss": cols["text_loss"][j][k],
                       "img_acc": cols["img_acc"][j][k], "text_acc": cols["text_acc"][j][k]}
                if traces[k] is not None:
                    traces[k].setdefault("stats", []).append(dict(rec, lr=lrs[k]))
                if loggers[k] is not None:
                    loggers[k].log({"train/image_loss": rec["image_loss"], "train/text_loss": rec["text_loss"],
                                    "train/image_acc": rec["img_acc"], "train/text_acc": rec["text_acc"], "train/lr": lrs[k]})
        last = {name: col[-1] for name, col in cols.items()}
        pending.clear()

    def take(loaders, its, k, n):
        """Head k's next n batches of one modality: re-iterates the loader first when its epoch is over (drawing the
        base seed and, at the first batch, the sampler seed - the order fetch_next produces)."""
        if its[k].batches_left() == 0:
            its[k] = iter(loaders[k])
        return its[k].take_run(n)

    def left(loaders, its):
        b = its[0].batches_left()
        return b if b > 0 else len(loaders[0])

    max_chunk = 64
    # traces[0]["timing"] = {"warmup": W}: wall-clock seconds of iterations W.. (stream-synchronised on both sides,
    # including the read-back of their stats) land in traces[0]["timing"]["seconds"] - bench.py's end-to-end arm
    timing = traces[0].get("timing") if traces[0] is not None else None
    t_start = None
    i = 0
    while any(running):
        next_eval = i if i % eval_freq == 0 else (i // eval_freq + 1) * eval_freq
        last_iter = min(max_iters[k] for k in range(K) if running[k]) - 1
        n = min(next_eval, last_iter) - i + 1
        n = max(1, min(n, max_chunk, log_slots - i % log_slots))
        if timing is not None:
            if i < timing["warmup"]:
                n = min(n, timing["warmup"] - i)
            elif t_start is None:
                flush()
                torch.cuda.current_stream().synchronize()
                t_start = time.perf_counter()
        if has_img:
            n = min(n, left(image_loaders, img_it))
        if has_txt:
            n = min(n, left(text_loaders, txt_it))
        perms_i, perms_t, span_i, span_t = [None] * K, [None] * K, None, None
        for k in range(K):  # image then text per head: the order the reference's step draws in
            if has_img:
                perms_i[k], st, tot = take(image_loaders, img_it, k, n)
                assert span_i in (None, (st, tot)), "heads left lock step"
                span_i = (st, tot)
            if has_txt:
                perms_t[k], st, tot = take(text_loaders, txt_it, k, n)
                assert span_t in (None, (st, tot)), "heads left lock step"
                span_t = (st, tot)
        bs_i, bs_t = (il0.batch_size if has_img else 0), (tl0.batch_size if has_txt else 0)
        rows = [(min(bs_i, span_i[1] - j * bs_i) if has_img else 0, min(bs_t, span_t[1] - j * bs_t) if has_txt else 0)
                for j in range(n)]
        assert all(r[0] >= 0 and r[1] >= 0 and r[0] + r[1] > 0 for r in rows), rows
        lrs = []
        for j in range(n):
            lrs.append([sch.get_last_lr()[0] for sch in schedulers])
            for sch in schedulers:
                sch.step()
        for k in range(K):
            tr = traces[k]
            if tr is not None and tr.get("indices", True) and running[k]:
                for name, its, span, bs in (("img_idx", img_it, span_i, bs_i), ("txt_idx", txt_it, span_t, bs_t)):
                    if span is not None:
                        host = its[k].perm_host[span[0]:span[0] + span[1]]
                        tr.setdefault(name, []).extend(c.clone() for c in host.split(bs))
        act = list(running)
        group.run(perms_i if has_img else None, perms_t if has_txt else None, span_i[0] if has_img else 0,
                  span_t[0] if has_txt else 0, rows, lrs, alphas, act, slot0=i)
        for j in range(n):
            pending.append((i + j, lrs[j], act))
        i += n
        last_step = i - 1

        if last_step % eval_freq == 0:
            flush()
            heads = [k for k in range(K) if running[k]]
            # every head's evaluation is enqueued before anything is read back: one synchronisation per round
            # the same draw order per head as the sequential loop (val, then test): each head has its own generator
            with_test = [k for k in heads if test_loaders[k] is not None]
            if adapter:  # head by head (the adapter runs in fp32 inside validate_enqueue), all enqueued before one read-back
                s_img = group.image_scales()
                results = [validate_enqueue(models[k], val_loaders[k], s_img[k]) for k in heads]
                t_res = {k: validate_enqueue(models[k], test_loaders[k], s_img[k]) for k in with_test}
                snaps = None
            else:
                results = validate_group_enqueue(group, models, heads, lambda k: val_loaders[k])
                t_res = dict(zip(with_test, validate_group_enqueue(group, models, with_test, lambda k: test_loaders[k]))) if with_test else {}
                snaps = group.W.clone()
            tests = [t_res.get(k) for k in heads]
            losses = torch.cat([r[0] for r in results]).cpu().tolist()
            hits = torch.cat([r[1] for r in results]).cpu().tolist()
            for h, k in enumerate(heads):
                val_loss, val_acc = float(losses[h]), int(hits[h]) / results[h][2]
                testlog = ""
                if tests[h] is not None:
                    testlog = f" | Test Acc: {int(tests[h][1].item()) / tests[h][2]:.4f}"
                if outs[k]["val_acc"] is None or val_acc > outs[k]["val_acc"]:
                    if snaps is None:  # every state-dict key: head.weight, img_proj.weight, img_scale, txt_scale
                        best = {n_: v.detach().cpu().clone() for n_, v in models[k].state_dict().items()}
                    else:
                        best = {"head.weight": snaps[k, :group.C * group.D].view(group.C, group.D).cpu()}
                    outs[k].update(iter=last_step, val_acc=val_acc, val_loss=val_loss, model=best)
                    no_improve[k] = 0
                else:
                    no_improve[k] += 1
                if traces[k] is not None:
                    traces[k].setdefault("evals", []).append((last_step, val_loss, val_acc))
                if loggers[k] is not None:
                    loggers[k].log({"val/val_loss": val_loss, "val/val_acc": val_acc, "iter": last_step})
                print(f"[{tags[k]}] Iter {last_step} | Img Loss: {last['image_loss'][k]:.4f} | "
                      f"Text Loss: {last['text_loss'][k]:.4f} | Img Acc: {last['img_acc'][k]:.4f} | "
                      f"Text Acc: {last['text_acc'][k]:.4f} | Val Loss: {val_loss:.4f} | Val Acc {val_acc:.4f}{testlog} | "
                      f"Count {no_improve[k]}/{patience[k]}")
                if no_improve[k] >= patience[k]:
                    print(f"=> [{tags[k]}] Early stopping at Iter {last_step}")
                    running[k] = False
        for k in range(K):
            if running[k] and i >= max_iters[k]:
                running[k] = False
    flush()
    if timing is not None and t_start is not None:
        torch.cuda.current_stream().synchronize()
        timing["seconds"], timing["iters"] = time.perf_counter() - t_start, i - timing["warmup"]
    for k in range(K):
        extra = {n_: v for n_, v in models[k].state_dict().items() if n_ not in outs[k]["model"]}
        models[k].load_state_dict({**extra, **outs[k]["model"]})
        val_loss, val_acc = validate(models[k], val_loaders[k], device=device)
        if loggers[k] is not None:
            loggers[k].log({"val/best_val_loss": val_loss, "val/best_val_acc": val_acc, "iter": outs[k]["iter"]})
        print(f"=> [{tags[k]}] Best Val Loss {val_loss:.4f}, Val Acc {val_acc:.4f} at Iter {outs[k]['iter']}")
    return outs


# ------------------------------------------------------------------------------------------------
# orchestration
# ------------------------------------------------------------------------------------------------

class _NullLogger:
    def log(self, *_a, **_k):
        pass


def setup_wandb_logger(hparams, args):
    """wandb when it is importable and not disabled, else a no-op (the reference calls wandb.init
    unconditionally, finetune.py:318-321, which needs network access)."""
    if os.environ.get("WANDB_MODE", "disabled") in ("disabled", "offline") and not os.environ.get("UML_WANDB"):
        return _NullLogger()
    import wandb
    return wandb.init(entity="unpaired_multimodal", project="unpaired_multimodal",
                      tags=[args.dataset, args.modality, args.hyperparams], config={**vars(args), **dict(hparams)},
                      reinit="finish_previous")


def _prepare(datasets, hparams, args, rng=None):
    """What ``setup`` does before the loop (finetune.py:323-384 of the reference): checkpoint directory, model,
    zero-shot initialisation, optimizer, scheduler, loaders.  Returns ``{"done": stored result}`` when the run's
    ``test_result.pth`` already exists.  ``rng``: generator the run's loaders draw their seeds from instead of the
    global one (batched sweeps)."""
    logger = setup_wandb_logger(hparams, args)
    device = args.device
    ckpt_dir = os.path.join(args.savepath, hparam_str(hparams["optim"], hparams["lr"], hparams["weight_decay"],
                                                      hparams["batch_size"], hparams["max_iter"], hparams["dropout"],
                                                      hparams["learnable_temp"]))
    makedirs(ckpt_dir)
    test_path = os.path.join(ckpt_dir, "test_result.pth")
    if os.path.exists(test_path) and not FLAG:
        print(f"=> Skipping {ckpt_dir} as it already exists!")
        return {"done": torch.load(test_path, map_location=device)}
    print(f"=> Setting up {ckpt_dir}")
    freeze = args.hyperparams == "linear"
    if args.use_clip:
        model = UMLClip(f"{args.clip_encoder}:{args.img_indim}", args.nclasses, logit_scale_init=args.logit, bias=False,
                        learnable_temp=hparams["learnable_temp"], freeze_backbone=freeze)
    else:
        shared = args.text_indim if args.modality == "crossmodal" else args.common_dim
        model = UML(f"{args.vision_model}:{args.img_indim}", shared, args.nclasses, bias=False,
                    learnable_temp=hparams["learnable_temp"], freeze_backbone=freeze)
    model.precision = getattr(args, "precision", "auto")
    model.to(device)
    print(f"=> UML trainable parameters: {sum(p.numel() for p in model.parameters())}")
    if args.classifier_init == "zeroshot" and (args.modality == "crossmodal" or
                                               (args.modality == "image" and args.common_dim == args.text_indim)):
        model.zero_shot_init(datasets["text_ds"])
    model.to(device)

    optimizer = build_optimizer(model.parameters(), hparams["optim"], hparams["lr"], hparams["weight_decay"])
    scheduler = build_lr_scheduler(optimizer, hparams["lr_scheduler"], hparams["warmup_iter"], hparams["max_iter"],
                                   warmup_type=hparams["warmup_type"], warmup_lr=hparams["warmup_min_lr"])
    bs, nw = hparams["batch_size"], args.num_workers
    rank, world = _dist()
    if world > 1 and getattr(args, "dp_sampler", "global") == "sharded":
        # per-rank sampler: every rank keeps and shuffles only its strided row shard; bs stays the GLOBAL batch size
        from .engine.datasets.utils import shard_bank
        ib, tb = datasets["img_tr_bank"], datasets["text_bank"]
        image_loader = BankLoader(shard_bank(ib.features, ib.labels, rank, world, device), -(-bs // world), shuffle=True,
                                  num_workers=nw, shard_of=(rank, world))
        text_loader = BankLoader(shard_bank(tb.features, tb.labels, rank, world, device), -(-bs // world), shuffle=True,
                                 num_workers=nw, shard_of=(rank, world))
    else:
        image_loader = BankLoader(datasets["img_tr_bank"], bs, shuffle=True, drop_last=False, num_workers=nw, rng=rng)
        text_loader = BankLoader(datasets["text_bank"], bs, shuffle=True, drop_last=False, num_workers=nw, rng=rng)
    if args.modality == "image":
        text_loader = None
        print("=> Running Unimodal: Image Only Model")
    elif args.modality == "text":
        image_loader = None
        print("=> Running Unimodal: Text Only Model")
    val_loader = BankLoader(datasets["img_val_bank"], bs, shuffle=False, num_workers=nw, rng=rng)
    test_loader = BankLoader(datasets["img_te_bank"], bs, shuffle=False, num_workers=nw, rng=rng)
    return dict(model=model, optimizer=optimizer, scheduler=scheduler, image_loader=image_loader, text_loader=text_loader,
                val_loader=val_loader, test_loader=test_loader, logger=logger, ckpt_dir=ckpt_dir, test_path=test_path,
                hparams=hparams)


def _finish(ctx, result, args):
    """The tail of ``setup`` (finetune.py:386-403): test accuracy of the restored best state, ``test_result.pth``."""
    test_loss, test_acc = validate(ctx["model"], ctx["test_loader"], device=args.device)
    ctx["model"] = None
    ctx["logger"].log({"test/test_loss": test_loss, "test/test_acc": test_acc})
    test_dict = {"test_acc": test_acc, "val_acc": result["val_acc"], "model": result["model"], "iter": result["iter"]}
    print(f"=> Test Acc: {test_acc:.4f}")
    if (not FLAG or getattr(args, "overwrite", False)) and _dist()[0] == 0:  # replicas are identical: rank 0 writes
        print(f"=> Saving Test Results for hparams to {ctx['test_path']}")
        torch.save(test_dict, ctx["test_path"])
    return test_dict


def setup(datasets, hparams, args):
    ctx = _prepare(datasets, hparams, args)
    if "done" in ctx:
        return ctx["done"]
    result = train(ctx["model"], ctx["image_loader"], ctx["text_loader"], ctx["val_loader"],
                   ctx["test_loader"] if args.eval_test else None, ctx["optimizer"], ctx["scheduler"], device=args.device,
                   max_iters=hparams["max_iter"], alpha=args.alpha, eval_freq=EVAL_FREQ, patience=hparams["patience"],
                   capture_features_during_training=False, features_pth=ctx["ckpt_dir"], args=args, logger=ctx["logger"])
    return _finish(ctx, result, args)


def run_seed(args, n):
    """Sampler seed of combination ``n`` of a batched sweep: a function of --seed, --alpha and the combination's position
    in the preset's grid only, so a combination's result does not depend on which others train with it."""
    return args.seed * 1000003 + n + 7919 * int(round(float(args.alpha) * 1000))


def setup_group(datasets, combos, args, positions=None):
    """``setup`` for several hyper-parameter combinations at once: the runs that can share a HeadGroup (same shapes,
    optimizer kind, batch size; no adapter, fixed temperatures) train in lock step (``train_group``), the rest one
    after the other.  ``args`` is one namespace for all combinations or a list with one per combination (runs that
    differ in --alpha and therefore in ``savepath``).  Run k's loaders draw from their own generator seeded
    ``run_seed(args_k, positions[k])`` (``positions``: each combination's index in the preset's grid, default
    0, 1, ...) - or from the global stream when ``args.seed < 0``."""
    from .engine.sweep import MAX_HEADS, adapter_group_blockers, group_blockers

    per_run = list(args) if isinstance(args, (list, tuple)) else [args] * len(combos)
    positions = list(positions) if positions is not None else list(range(len(combos)))
    args = per_run[0]
    with_adapters = bool(getattr(args, "sweep_batched_adapter", False))

    def blockers(cand):
        """--sweep-batched-adapter: runs with an image adapter or learnable temperatures form AdapterHeadGroups."""
        ms = [ctxs[c]["model"] for c in cand]
        adapter = with_adapters and any(m.img_proj is not None or getattr(m, "learnable_temp", False) for m in ms)
        return (adapter_group_blockers if adapter else group_blockers)(
            ms, [ctxs[c]["optimizer"] for c in cand], [ctxs[c]["image_loader"] for c in cand],
            [ctxs[c]["text_loader"] for c in cand])

    results = [None] * len(combos)
    ctxs = {}
    for n, hp in enumerate(combos):
        a = per_run[n]
        print(f"=> Preparing {n + 1}/{len(combos)}: alpha {a.alpha} {hp}")
        seed = run_seed(a, positions[n]) if a.seed >= 0 else int(torch.empty((), dtype=torch.int64).random_().item())
        ctx = _prepare(datasets, hp, a, rng=torch.Generator().manual_seed(seed))
        if "done" in ctx:
            results[n] = ctx["done"]
        else:
            ctx["args"] = a
            ctxs[n] = ctx
    todo = sorted(ctxs)
    while todo:
        # greedy grouping: everything compatible with the first open run joins it
        first, members = todo[0], [todo[0]]
        for n in todo[1:]:
            if len(members) >= MAX_HEADS:
                break
            cand = members + [n]
            if not blockers(cand):
                members = cand
        solo = blockers([first]) or _dist()[1] > 1
        todo = [n for n in todo if n not in members]
        col = lambda key: [ctxs[c][key] for c in members]
        if solo:  # not batchable at all (adapter, learnable temperature, data parallel): the plain loop, same loaders
            c = ctxs[first]
            outs = [train(c["model"], c["image_loader"], c["text_loader"], c["val_loader"],
                          c["test_loader"] if args.eval_test else None, c["optimizer"], c["scheduler"],
                          device=args.device, max_iters=c["hparams"]["max_iter"], alpha=c["args"].alpha,
                          eval_freq=EVAL_FREQ, patience=c["hparams"]["patience"], args=c["args"], logger=c["logger"])]
        else:
            print(f"=> Training {len(members)} combinations in lock step: {members}")
            outs = train_group(col("model"), col("image_loader"), col("text_loader"), col("val_loader"),
                               col("test_loader") if args.eval_test else None, col("optimizer"), col("scheduler"),
                               device=args.device, max_iters=[ctxs[c]["hparams"]["max_iter"] for c in members],
                               alphas=[ctxs[c]["args"].alpha for c in members], eval_freq=EVAL_FREQ,
                               patience=[ctxs[c]["hparams"]["patience"] for c in members], loggers=col("logger"),
                               tags=[f"run {c + 1}" for c in members])
        for c, out in zip(members, outs):
            ctx = ctxs.pop(c)
            results[c] = _finish(ctx, out, ctx["args"])
    return results


def _grid(hyperparams):
    grid = {k: (v if isinstance(v, list) else [v]) for k, v in hyperparams.items()}
    keys = list(grid)
    return [dict(zip(keys, combo)) for combo in product(*[grid[k] for k in keys])]


def _collect(hps, outcomes, args):
    """The bookkeeping of the reference's ``sweep`` (finetune.py:417-448) over finished runs: running best, results.pth,
    the final summary."""
    results = {"test_acc": [], "val_acc": [], "hparams": [], "model_records": []}
    best_val = best_test = 0
    best_hp = None
    for n, (hp, res) in enumerate(zip(hps, outcomes)):
        print(f"=> Running {n + 1}/{len(hps)}: {hp}")
        if callable(res):
            res = res()
        results["test_acc"].append(res["test_acc"])
        results["val_acc"].append(res["val_acc"])
        results["hparams"].append(hp)
        if res["val_acc"] > best_val:
            best_val, best_test, best_hp = res["val_acc"], res["test_acc"], hp
            print(f"=> New Best Val Acc: {best_val:.4f} | Test Acc: {best_test:.4f}")
        print(f"=> Best Val Acc (so far): {best_val:.4f} | Test Acc (corresponding): {best_test:.4f}")
        print(f"=> Best Hyperparameters (so far): {best_hp}")
        print("--------------------------------------------------------\n")
    if (not FLAG or getattr(args, "overwrite", False)) and _dist()[0] == 0:
        print(f"=> Saving results across all hparams to {args.savepath}")
        torch.save(results, os.path.join(args.savepath, "results.pth"))
    k = int(torch.argmax(torch.tensor(results["val_acc"])))
    print(f"=> [FINAL] Best Val Acc: {results['val_acc'][k]:.4f} | Best Test Acc: {results['test_acc'][k]:.4f}")
    print(f"=> [FINAL] Mean Val Acc: {torch.tensor(results['val_acc']).mean():.4f} | "
          f"Mean Test Acc: {torch.tensor(results['test_acc']).mean():.4f}")
    print(f"=> [FINAL] Best Hyperparameters: {results['hparams'][k]}")
    return results, results["val_acc"][k], results["test_acc"][k]


def sweep(datasets, hyperparams, args):
    hps = _grid(hyperparams)
    if getattr(args, "sweep_batched", False) or getattr(args, "sweep_batched_adapter", False):
        # --sweep-batched: the combinations train in lock step on one GPU (setup_group) instead of one after the other
        return _collect(hps, setup_group(datasets, hps, args), args)
    return _collect(hps, [lambda hp=hp: setup(datasets, hp, args) for hp in hps], args)


def sweep_alphas(datasets, hyperparams, args_per_alpha):
    """``sweep`` for several values of --alpha at once.  The reference's YAML lists alpha (configs/finetune.yaml:17) and
    runs ``main`` once per value over the same banks; here all alpha x hyper-parameter combinations (<= 32 per
    HeadGroup) train in lock step.  ``args_per_alpha``: one namespace per alpha (own ``alpha`` and ``savepath``).
    Result files land where one ``main`` per alpha would have put them; returns ``[sweep's return value per alpha]``."""
    hps = _grid(hyperparams)
    runs, owners = [], []
    for a in args_per_alpha:
        runs += hps
        owners += [a] * len(hps)
    outcomes = setup_group(datasets, runs, owners, positions=[n % len(hps) for n in range(len(runs))])
    return [_collect(hps, outcomes[i * len(hps):(i + 1) * len(hps)], a) for i, a in enumerate(args_per_alpha)]


def main(args, alphas=None):
    """``alphas``: several --alpha values to train in ONE batched sweep over the banks loaded once (``sweep_alphas``; the
    reference runs ``main`` once per alpha of its YAML list).  Returns ``sweep``'s triple, or a list of them (one per
    alpha) when ``alphas`` is given."""
    if args.seed >= 0:
        print("=> Setting fixed seed: {}".format(args.seed))
        set_random_seed(args.seed)
    if not torch.cuda.is_available():
        raise RuntimeError("uml_b200.finetune needs a CUDA device: the hot path has no CPU implementation")
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    args.device = f"cuda:{local_rank}"
    torch.cuda.set_device(local_rank)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and not torch.distributed.is_initialized():
        # launched with torchrun: one rank per GPU, data parallel over the rows of every batch (DESIGN.md section 6)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=torch.device(args.device))
    args.use_clip = args.vision_model == "" and args.language_model == ""
    if getattr(args, "sweep_batched_adapter", False):
        args.sweep_batched = True
    encoder_name = args.clip_encoder if args.use_clip else f"{args.vision_model}-{args.language_model}"
    alpha_list = [float(a) for a in alphas] if alphas else [args.alpha]
    savepaths = [savedir(args.result_dir, args.dataset, encoder_name, args.train_shot, args.seed, args.text_type,
                         args.text_shot, args.image_augmentation, args.modality, args.classifier_init, a,
                         getattr(args, "text_batch_size", 0), args.custom_name, args) for a in alpha_list]
    args.savepath = savepaths[0]
    for sp in savepaths:
        makedirs(sp)
    logfiles = [open(os.path.join(sp, "log.txt"), "w") for sp in dict.fromkeys(savepaths)]
    prev_stdout = sys.stdout  # (the caller's redirection - pytest capture, a notebook, an outer Tee - stays in the chain)
    sys.stdout = Tee(prev_stdout, *logfiles)
    try:
        print("=> Arguments:", args)
        text_encoder = args.clip_encoder if args.use_clip else args.language_model
        text_path = text_outdir(args.feature_dir, text_encoder, args.dataset, args.text_type)
        print(f"=> Loading text features from: {text_path}")
        tf = load_text_bank(text_path)
        shots = args.text_shot
        if shots is not None and shots != "average":
            shots = int(shots)
        # a v2 file next to the v1 text bank (features.convert_bank) carries the class-sorted row index: the per-class
        # selection / averaging then walks it instead of masking the labels once per class
        text_ds = TextTensorDataset(tf["features"], tf["labels"], tf["eot_indices"], n_shots=shots,
                                    class_order=tf.get("class_order"), class_starts=tf.get("class_starts"))

        image_encoder = args.clip_encoder if args.use_clip else args.vision_model
        tr_path = img_outdir(args.feature_dir, image_encoder, args.dataset, args.image_augmentation, args.train_shot,
                             args.seed, "train")
        te_path = img_outdir(args.feature_dir, image_encoder, args.dataset, args.image_augmentation, args.train_shot,
                             args.seed, "test")
        print(f"=> Loading image features from: {tr_path} and {te_path}")
        dev = args.device
        # v2 bank files next to the .pth ones (features.convert_bank) are mapped and streamed to HBM; else the v1 dicts
        tr_bank, tr_meta = load_feature_bank(tr_path, dev, "train")
        val_bank, _ = load_feature_bank(tr_path, dev, "val")
        te_bank, te_meta = load_feature_bank(te_path, dev)
        lab2cname = tr_meta.get("lab2cname") or te_meta.get("lab2cname") or tf.get("lab2cname")
        args.img_indim = int(tr_bank.dim)
        args.text_indim = int(tf["features"].shape[1])
        if args.use_clip and args.img_indim != args.text_indim:
            raise ValueError("CLIP image and text features must share a width")
        args.nclasses = len(lab2cname) if lab2cname else int(max(tr_bank.labels.max(), te_bank.labels.max())) + 1
        datasets = {
            "text_ds": text_ds, "text_bank": FeatureBank.from_text_dataset(text_ds, dev),
            "img_tr_bank": tr_bank, "img_val_bank": val_bank, "img_te_bank": te_bank,
        }
        if alphas:
            import copy
            per_alpha = []
            for a, sp in zip(alpha_list, savepaths):
                c = copy.copy(args)
                c.alpha, c.savepath = a, sp
                per_alpha.append(c)
            out = sweep_alphas(datasets, HYPER_DICT[args.hyperparams], per_alpha)
        else:
            out = sweep(datasets, HYPER_DICT[args.hyperparams], args)
        del datasets
        print("Done!")
    finally:
        sys.stdout = prev_stdout
        for f in logfiles:
            f.close()
    return out


def cli(argv=None):
    import yaml

    outer = argparse.ArgumentParser(description="UML fine-tuning over feature banks")
    outer.add_argument("-c", "--config", type=str, default="config.yaml", help="Configuration file")
    outer.add_argument("-s", "--slurm", action="store_true", help="Launched with slurm")
    outer.add_argument("-d", "--debug", action="store_true", help="Debug mode")
    outer.add_argument("-f", "--flag", action="store_true", help="Run despite existing experiments directory")
    outer.add_argument("-o", "--overwrite", action="store_true", help="Overwrite existing experiments directory")
    outer_args, rest = outer.parse_known_args(argv)
    global FLAG
    FLAG = int(outer_args.flag)
    if outer_args.debug:
        args = parser.parse_args(rest)
        args.overwrite = outer_args.overwrite
        return main(args)
    with open(outer_args.config) as f:
        sweep_args = yaml.load(f, Loader=yaml.FullLoader)
    keys = list(sweep_args)
    combos = [dict(zip(keys, v)) for v in product(*[(v if isinstance(v, list) else [v]) for v in sweep_args.values()])]
    print("Total combinations:", len(combos))
    for i, c in enumerate(combos):
        print(f"Combination {i}: {c}")
    if outer_args.slurm:
        job = int(os.getenv("SLURM_ARRAY_TASK_ID", "-1"))
        if not 0 <= job < len(combos):
            print("Invalid SLURM_ARRAY_TASK_ID")
            sys.exit(1)
        combos = [combos[job]]
    # sweep_batched: jobs that differ only in alpha share their banks, so they become ONE job whose alpha x
    # hyper-parameter combinations train in lock step (main(args, alphas=[...]))
    jobs = []
    for c in combos:
        rest_ = {k: v for k, v in c.items() if k != "alpha"}
        batched = c.get("sweep_batched") or c.get("sweep_batched_adapter")
        mate = next((j for j in jobs if batched and j[0] == rest_ and "alpha" in c), None)
        if mate is not None:
            mate[1].append(c["alpha"])
        else:
            jobs.append((rest_, [c["alpha"]] if "alpha" in c else []))
    for i, (c, alphas_) in enumerate(jobs):
        print(f"=> Running job {i}")
        if alphas_:
            c = dict(c, alpha=alphas_[0])
        args = parser.parse_args([], argparse.Namespace(**c))
        args.overwrite = outer_args.overwrite
        if len(alphas_) > 1:
            main(args, alphas=alphas_)
        else:
            main(args)


if __name__ == "__main__":
    cli()
