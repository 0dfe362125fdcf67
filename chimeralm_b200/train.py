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

import logging
from collections import OrderedDict
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


def fit(engine, seqs, labels, *, epochs: int = 3, batch_size: int = 32, seed: int = 0, lr: float = 1e-3,
        weight_decay: float = 0.01, dropout: float = 0.1, log_every: int = 0) -> list[float]:
    """Train the head of `engine` on (seqs, labels): per epoch the length-bucketed batches run in an order shuffled by
    `seed` and the epoch.  Returns the mean loss of every epoch."""
    labels = np.asarray(labels, np.int64)
    lens = np.array([len(s) for s in seqs], np.int64)
    batches = make_batches(lens, batch_size)
    max_b = max(len(b) for b in batches)
    max_t = max(int(lens[b].max()) + 1 for b in batches)
    engine.reserve(max_b, max_t, max(len(b) * (int(lens[b].max()) + 1) for b in batches))
    engine.head_train_begin(lr=lr, weight_decay=weight_decay, dropout=dropout, seed=seed)
    history = []
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
    return history


def tuned_state_dict(base_sd, engine) -> "OrderedDict[str, torch.Tensor]":
    """`base_sd` with its head tensors replaced by the engine's trained ones; every other tensor is the input's own."""
    head = engine.head_state_dict()
    out = OrderedDict()
    for k, v in base_sd.items():
        out[k] = head[k].reshape(v.shape).clone() if k in head else v
    return out


def finetune(data_path, ckpt_path, output_path, *, epochs: int = 3, lr: float = 1e-3, batch_size: int = 32,
             seed: int = 0, seed_weights: int = 0, device: int = 0, weight_decay: float = 0.01,
             dropout: float = 0.1) -> list[float]:
    """The `finetune` command: labelled reads -> trained head -> Lightning-layout checkpoint at `output_path`."""
    from .engine import Engine

    sd = load_checkpoint(ckpt_path) if ckpt_path is not None else make_state_dict(seed_weights)
    if not any(k.startswith(BACKBONE_PREFIX) for k in sd):
        raise ValueError("the checkpoint holds no backbone tensors (net.backbone.backbone.*)")
    _, seqs, labels = read_labelled(data_path)
    log.info(f"{len(seqs)} labelled reads ({int(labels.sum())} with label 1)")
    eng = Engine(sd, device=device, max_batch=2, max_tokens=1024)   # fit() reserves for its batches
    try:
        history = fit(eng, seqs, labels, epochs=epochs, batch_size=batch_size, seed=seed, lr=lr,
                      weight_decay=weight_decay, dropout=dropout)
        out = tuned_state_dict(sd, eng)
    finally:
        eng.close()
    assert all(torch.equal(out[k], sd[k]) for k in sd if not k.startswith(HEAD_PREFIX))
    Path(output_path).parent.mkdir(parents=True, exist_ok=True)
    save_lightning_ckpt(out, output_path)
    return history
