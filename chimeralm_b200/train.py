"""Fine-tuning of the classification head on labelled reads, with the backbone frozen.

The reference trains through `ClassificationLit.training_step` / `model_step` (cross-entropy on `net(input_ids)`,
chimeralm/models/basic_module.py:87-104) with AdamW (`configure_optimizers`, :200-223) and reads a read's label from the
`|0` / `|1` suffix of its id (`parse_target`, chimeralm/data/tokenizer.py:25-33).  Here one optimizer step is one call of
`clm_head_train_step` (csrc/head_train.cuh): the forward is the unchanged predict forward, the head's backward and the
AdamW update run on the GPU; the backbone's weights are never written.

Host side only: label parsing, the numpy mirror of the dropout masks (what the parity tests compare against), batching
and the epoch loop.
"""

from __future__ import annotations

import json
import logging
from collections import OrderedDict
from dataclasses import dataclass
from pathlib import Path

import numpy as np
import torch

from . import synth
from .weights import BACKBONE_PREFIX, HEAD_PREFIX, load_checkpoint, make_state_dict, save_lightning_ckpt

log = logging.getLogger("chimeralm")

MAX_BASES = 32768                     # a read is cut to its first 32 768 bases (+ [SEP] = the model's 32 769 tokens)
HEAD_HIDDEN = 512
DROPOUT_SITES = ("classifier.2", "classifier.5", "classifier.6.layers.2")


def parse_target(name: str) -> int | None:
    """Label of a training read from its id `name|label` (the suffix the reference's `addtarget` tool appends and
    `parse_target` reads): the integer after the last `|`.  An id without a `|` has no label: None."""
    head, sep, tail = name.rpartition("|")
    if not sep:
        return None
    try:
        return int(tail)
    except ValueError:
        return None


# ------------------------------------------------------------------------------------------
# Dropout keep-masks: bit-exact mirror of dropout_keep() in csrc/head_train.cuh

_M32 = np.uint64(0xFFFFFFFF)


def _mix32(x: np.ndarray) -> np.ndarray:
    x = x.astype(np.uint64) & _M32
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x7FEB352D)) & _M32
    x ^= x >> np.uint64(15)
    x = (x * np.uint64(0x846CA68B)) & _M32
    x ^= x >> np.uint64(16)
    return x


def dropout_threshold(p: float) -> int:
    """keep <=> (hash >> 8) >= round(p * 2^24)."""
    return int(np.floor(p * 16777216.0 + 0.5))


def dropout_keep(seed: int, step: int, site: int, read, unit, p: float) -> np.ndarray:
    """Keep bits of the dropout masks (broadcast over `read` and `unit`) exactly as the device draws them."""
    read, unit = np.broadcast_arrays(np.asarray(read, np.uint64), np.asarray(unit, np.uint64))
    h = _mix32(np.full(read.shape, (int(seed) & 0xFFFFFFFF) ^ 0x9E3779B9, np.uint64))
    h = _mix32(h ^ np.uint64(int(step) & 0xFFFFFFFF))
    h = _mix32(h ^ np.uint64(site))
    h = _mix32(h ^ read)
    h = _mix32(h ^ unit)
    return (h >> np.uint64(8)) >= np.uint64(dropout_threshold(p))


def dropout_masks(seed: int, step: int, B: int, p: float, hidden: int = HEAD_HIDDEN) -> np.ndarray:
    """bool [3, B, hidden]: the keep-masks of the three dropout sites (DROPOUT_SITES) for training call `step`."""
    b = np.arange(B, dtype=np.uint64)[:, None]
    u = np.arange(hidden, dtype=np.uint64)[None, :]
    return np.stack([dropout_keep(seed, step, s, b, u, p) for s in range(3)])


def adamw_update(p, g, m, v, t: int, lr: float, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.01):
    """One AdamW step in float32, the arithmetic of adamw_kernel (csrc/head_train.cuh) restated in numpy; `t` counts
    from 1.  Returns the new (p, m, v)."""
    f = np.float32
    p, g, m, v = (np.asarray(a, f) for a in (p, g, m, v))
    b1, b2 = f(betas[0]), f(betas[1])
    step_size = f(lr / (1.0 - betas[0] ** t))
    bc2_sqrt = f(np.sqrt(1.0 - betas[1] ** t))
    p = p * (f(1) - f(lr) * f(weight_decay))
    m = m + (f(1) - b1) * (g - m)
    v = v * b2 + (f(1) - b2) * g * g
    p = p - step_size * m / (np.sqrt(v) / bc2_sqrt + f(eps))
    return p, m, v


# ------------------------------------------------------------------------------------------
# Labelled input and batches

def read_labelled(path, max_bases: int = MAX_BASES):
    """(names, uint8 base arrays, int64 labels) of a FASTQ(.gz) or Parquet file whose ids carry `|0` / `|1`."""
    from .data import read_fastq_bytes, read_parquet_records

    path = Path(path)
    recs = read_parquet_records(path) if path.suffix == ".parquet" else read_fastq_bytes(path)
    names, seqs, labels = [], [], []
    for name, seq in recs:
        y = parse_target(name)
        if y not in (0, 1):
            raise ValueError(f"read '{name}' has no 0/1 label: training ids must end in '|0' or '|1'")
        names.append(name)
        seqs.append(seq[:max_bases])
        labels.append(y)
    if not names:
        raise ValueError(f"{path}: no reads")
    return names, seqs, np.asarray(labels, np.int64)


def make_batches(lengths: np.ndarray, batch_size: int) -> list[np.ndarray]:
    """Reads sorted by length and cut into batches of <= batch_size (synth.bucket_batches): little padding per batch."""
    return synth.bucket_batches(np.asarray(lengths, np.int64), batch_size)


def pack_batch(engine, seqs, idx) -> torch.Tensor:
    """Token ids of the reads `idx` on the engine's device: ids + [SEP], left-padded to the longest (what `predict` feeds)."""
    from .engine import pack_reads

    chosen = [seqs[i] for i in idx]
    T = max(len(s) for s in chosen) + 1
    bases, offs = pack_reads([s.tobytes() for s in chosen])
    ids, _ = engine.encode(bases, offs, T, add_cls=False, add_sep=True, pad_left=True, max_bases=MAX_BASES)
    return ids


# ------------------------------------------------------------------------------------------
# Evaluation on labelled reads (the reference's validation / test steps and their torchmetrics)

def cross_entropy_rows(logits, targets) -> np.ndarray:
    """Per-read cross-entropy of logits [B,2] against 0/1 targets, in float64: lse - l_y with the max subtracted
    first (ce_row of csrc/head_train.cuh in double precision)."""
    lg = np.asarray(logits, np.float64)
    y = np.asarray(targets, np.int64)
    m = lg.max(axis=1)
    lse = m + np.log(np.exp(lg[:, 0] - m) + np.exp(lg[:, 1] - m))
    return lse - lg[np.arange(len(y)), y]


def auroc(targets, prob) -> float | None:
    """Area under the ROC curve of `prob` as the score of class 1, from ranks (Mann-Whitney U): the fraction of
    (positive, negative) pairs in which the positive read has the higher probability, a tie counting one half.  None
    when one class is absent."""
    y = np.asarray(targets, np.int64)
    p = np.asarray(prob, np.float64)
    n_pos = int((y == 1).sum())
    n_neg = len(y) - n_pos
    if n_pos == 0 or n_neg == 0:
        return None
    order = np.argsort(p, kind="stable")
    sp = p[order]
    starts = np.flatnonzero(np.r_[True, sp[1:] != sp[:-1]])   # first position of every run of equal probabilities
    ends = np.r_[starts[1:], len(sp)]
    ranks = np.empty(len(p), np.float64)
    ranks[order] = np.repeat((starts + ends + 1) / 2.0, ends - starts)   # 1-based ranks, ties share their mean
    return float((ranks[y == 1].sum() - n_pos * (n_pos + 1) / 2.0) / (n_pos * n_neg))


def binary_metrics(targets, preds, prob, loss) -> dict:
    """Metrics of a labelled set on the host in float64, class 1 (chimera artefact) positive:
    loss       mean per-read cross-entropy (a mean over reads, not over batches)
    accuracy   (tp + tn) / n
    precision  tp / (tp + fp),  recall  tp / (tp + fn),  f1  2 tp / (2 tp + fp + fn)  (0 when the denominator is 0)
    auroc      `auroc` (None with one class only)
    confusion  [[tn, fp], [fn, tp]]: rows are targets, columns predictions"""
    y = np.asarray(targets, np.int64)
    yhat = np.asarray(preds, np.int64)
    loss = np.asarray(loss, np.float64)
    n = len(y)
    if n == 0 or not (len(yhat) == len(loss) == len(np.asarray(prob)) == n):
        raise ValueError("binary_metrics: targets, preds, prob and loss must be non-empty and of one length")
    tp = int(((y == 1) & (yhat == 1)).sum())
    tn = int(((y == 0) & (yhat == 0)).sum())
    fp = int(((y == 0) & (yhat == 1)).sum())
    fn = int(((y == 1) & (yhat == 0)).sum())

    def ratio(a, b):
        return a / b if b else 0.0

    return {"reads": n, "loss": float(loss.mean()), "accuracy": (tp + tn) / n, "precision": ratio(tp, tp + fp),
            "recall": ratio(tp, tp + fn), "f1": ratio(2 * tp, 2 * tp + fp + fn), "auroc": auroc(y, prob),
            "confusion": [[tn, fp], [fn, tp]]}


def evaluate(engine, seqs, labels, batch_size: int = 32):
    """Score the head of `engine` on labelled reads: the batches training forms (`make_batches`, `pack_batch`), one
    `eval_step` each.  Returns (binary_metrics, per-read {"label", "prob", "loss"} in input order)."""
    labels = np.asarray(labels, np.int64)
    lens = np.array([len(s) for s in seqs], np.int64)
    batches = make_batches(lens, batch_size)
    engine.reserve(max(len(b) for b in batches), max(int(lens[b].max()) + 1 for b in batches),
                   max(len(b) * (int(lens[b].max()) + 1) for b in batches))
    n = len(seqs)
    pred, prob, loss = np.zeros(n, np.int64), np.zeros(n, np.float32), np.zeros(n, np.float32)
    for idx in batches:
        _, lab, ce, p = engine.eval_step(pack_batch(engine, seqs, idx), torch.from_numpy(labels[idx]))
        pred[idx], prob[idx], loss[idx] = lab.cpu().numpy(), p.cpu().numpy(), ce.cpu().numpy()
    return binary_metrics(labels, pred, prob, loss), {"label": pred, "prob": prob, "loss": loss}


@dataclass
class Validation:
    """Validation of a training run: `records[k]` holds the metrics after epoch k (0 = before training), `best` the
    chosen epoch and `head` the trained tensors after it (the head's, and with `train_tail` the tail's too)."""
    records: list
    best: int
    head: dict
    stopped_early: bool


def best_epoch(records) -> int:
    """The epoch (>= 1) to keep: the highest validation F1, ties to the lower validation loss, then to the earlier
    epoch.  Epoch 0 (before training) is never chosen.  0 when no epoch has been trained."""
    trained = [r for r in records if r["epoch"] >= 1]
    if not trained:
        return 0
    return min(trained, key=lambda r: (-r["f1"], r["loss"], r["epoch"]))["epoch"]


def epochs_without_improvement(records) -> int:
    """Trained epochs since the last that raised the best validation F1 (the first trained epoch always does): early
    stopping with patience N stops once this reaches N."""
    best, since = -np.inf, 0
    for r in records:
        if r["epoch"] < 1:
            continue
        if r["f1"] > best:
            best, since = r["f1"], 0
        else:
            since += 1
    return since


def _validate(engine, val, batch_size, epoch, train_loss) -> dict:
    metrics, _ = evaluate(engine, val[0], val[1], batch_size)
    rec = {"epoch": epoch, "train_loss": train_loss, **metrics}
    auc = "n/a" if rec["auroc"] is None else f"{rec['auroc']:.4f}"
    when = "before training" if epoch == 0 else f"after epoch {epoch}"
    log.info(f"validation {when}: loss {rec['loss']:.4f} accuracy {rec['accuracy']:.4f} "
             f"precision {rec['precision']:.4f} recall {rec['recall']:.4f} F1 {rec['f1']:.4f} AUROC {auc}")
    return rec


def trained_state_dict(engine, train_tail: bool) -> dict:
    """The tensors a run trains, as they stand: the head's, and with `train_tail` the last block's tail and ln_f."""
    out = dict(engine.head_state_dict())
    if train_tail:
        out.update(engine.tail_state_dict())
    return out


def fit(engine, seqs, labels, *, epochs: int = 3, batch_size: int = 32, seed: int = 0, lr: float = 1e-3,
        weight_decay: float = 0.01, dropout: float = 0.1, log_every: int = 0, val=None, patience: int | None = None,
        train_tail: bool = False, tail_lr: float | None = None):
    """Train the head of `engine` on (seqs, labels): per epoch the length-bucketed batches run in an order shuffled by
    `seed` and the epoch.  Returns the mean loss of every epoch.  With `train_tail` the last block's tail (out_proj,
    norm2, fc1, fc2) and ln_f train together with the head, with learning rate `tail_lr` (default `lr`).

    With `val` = (seqs, labels) of held-out reads the head is evaluated (`evaluate`, dropout off) before training
    (epoch 0, reported only) and after every epoch, and `patience` stops training after that many epochs without a
    better validation F1.  Returns (losses, Validation) then: the records of every epoch, the chosen epoch
    (`best_epoch`) and the head's tensors after it."""
    if val is not None and epochs < 1:
        raise ValueError("validation needs at least one epoch")
    if tail_lr is not None and not train_tail:
        raise ValueError("tail_lr needs train_tail")
    labels = np.asarray(labels, np.int64)
    lens = np.array([len(s) for s in seqs], np.int64)
    batches = make_batches(lens, batch_size)
    max_b = max(len(b) for b in batches)
    max_t = max(int(lens[b].max()) + 1 for b in batches)
    engine.reserve(max_b, max_t, max(len(b) * (int(lens[b].max()) + 1) for b in batches))
    engine.head_train_begin(lr=lr, weight_decay=weight_decay, dropout=dropout, seed=seed)
    if train_tail:
        engine.tail_train_begin(lr if tail_lr is None else tail_lr)
    history = []
    if val is not None:
        run = Validation([], 0, {}, False)
        run.records.append(_validate(engine, val, batch_size, 0, None))
    for ep in range(epochs):
        order = np.random.default_rng([seed, ep]).permutation(len(batches))
        losses = []
        for k, bi in enumerate(order):
            idx = batches[bi]
            ids = pack_batch(engine, seqs, idx)
            loss = engine.head_train_step(ids, torch.from_numpy(labels[idx]))
            losses.append(float(loss))
            if log_every and (k + 1) % log_every == 0:
                log.info(f"epoch {ep + 1} batch {k + 1}/{len(batches)} loss {losses[-1]:.4f}")
        history.append(float(np.mean(losses)))
        log.info(f"epoch {ep + 1}/{epochs}: mean loss {history[-1]:.4f}")
        if val is not None:
            # the export also refreshes the forward's copy of attention.2.bias, so that the validation forward is the
            # forward of the saved checkpoint bit for bit
            head = trained_state_dict(engine, train_tail)
            run.records.append(_validate(engine, val, batch_size, ep + 1, history[-1]))
            if best_epoch(run.records) == ep + 1:
                run.best, run.head = ep + 1, head
            if patience is not None and epochs_without_improvement(run.records) >= patience and ep + 1 < epochs:
                run.stopped_early = True
                log.info(f"no better validation F1 for {patience} epochs: stopping after epoch {ep + 1}")
                break
    if val is None:
        return history
    log.info(f"chosen epoch {run.best}: validation F1 {run.records[run.best]['f1']:.4f}, "
             f"loss {run.records[run.best]['loss']:.4f}")
    return history, run


def tuned_state_dict(base_sd, engine, train_tail: bool = False) -> "OrderedDict[str, torch.Tensor]":
    """`base_sd` with its head tensors (and with `train_tail` the tail's) replaced by the engine's trained ones; every
    other tensor is the input's own."""
    return with_head(base_sd, trained_state_dict(engine, train_tail))


def with_head(base_sd, head) -> "OrderedDict[str, torch.Tensor]":
    """`base_sd` with the tensors named in `head` replaced (reshaped to the base's shapes)."""
    out = OrderedDict()
    for k, v in base_sd.items():
        out[k] = head[k].reshape(v.shape).clone() if k in head else v
    return out


def finetune(data_path, ckpt_path, output_path, *, epochs: int = 3, lr: float = 1e-3, batch_size: int = 32,
             seed: int = 0, seed_weights: int = 0, device: int = 0, weight_decay: float = 0.01,
             dropout: float = 0.1, val_path=None, patience: int | None = None, train_tail: bool = False,
             tail_lr: float | None = None) -> list[float]:
    """The `finetune` command: labelled reads -> trained head -> Lightning-layout checkpoint at `output_path`.
    With `train_tail` the last block's tail and ln_f train too (`fit`), and the checkpoint replaces those tensors as well.

    With `val_path` (labelled reads, `read_labelled`) the head is validated before training and after every epoch
    (`fit`); the checkpoint holds the head of the chosen epoch (`best_epoch`), and the records go to
    `<output_path>.val.json`.  `patience` (needs `val_path`) stops after that many epochs without a better F1."""
    from .engine import Engine, tail_keys

    if patience is not None and (val_path is None or patience < 1):
        raise ValueError("patience needs validation reads (--val) and must be >= 1")
    if tail_lr is not None and not train_tail:
        raise ValueError("--tail-lr needs --train-tail")
    sd = load_checkpoint(ckpt_path) if ckpt_path is not None else make_state_dict(seed_weights)
    if not any(k.startswith(BACKBONE_PREFIX) for k in sd):
        raise ValueError("the checkpoint holds no backbone tensors (net.backbone.backbone.*)")
    _, seqs, labels = read_labelled(data_path)
    log.info(f"{len(seqs)} labelled reads ({int(labels.sum())} with label 1)")
    val = None
    if val_path is not None:
        _, vseqs, vlabels = read_labelled(val_path)
        log.info(f"{len(vseqs)} validation reads ({int(vlabels.sum())} with label 1)")
        val = (vseqs, vlabels)
    eng = Engine(sd, device=device, max_batch=2, max_tokens=1024)   # fit() reserves for its batches
    try:
        if val is None:
            history = fit(eng, seqs, labels, epochs=epochs, batch_size=batch_size, seed=seed, lr=lr,
                          weight_decay=weight_decay, dropout=dropout, train_tail=train_tail, tail_lr=tail_lr)
            out = tuned_state_dict(sd, eng, train_tail)
        else:
            history, run = fit(eng, seqs, labels, epochs=epochs, batch_size=batch_size, seed=seed, lr=lr,
                               weight_decay=weight_decay, dropout=dropout, val=val, patience=patience,
                               train_tail=train_tail, tail_lr=tail_lr)
            out = with_head(sd, run.head)
        tail = set(tail_keys(eng.cfg.n_layer)) if train_tail else set()
    finally:
        eng.close()
    # every tensor that was not trained equals the input
    assert all(torch.equal(out[k], sd[k]) for k in sd if not (k.startswith(HEAD_PREFIX) or k in tail))
    Path(output_path).parent.mkdir(parents=True, exist_ok=True)
    save_lightning_ckpt(out, output_path)
    if val is not None:
        report = {"train": str(data_path), "val": str(val_path), "checkpoint": str(output_path), "batch_size": batch_size,
                  "best_epoch": run.best, "stopped_early": run.stopped_early, "patience": patience,
                  "epochs": run.records}
        Path(str(output_path) + ".val.json").write_text(json.dumps(report, indent=1) + "\n")
        log.info(f"validation records saved to {output_path}.val.json; the checkpoint holds epoch {run.best}")
    return history
