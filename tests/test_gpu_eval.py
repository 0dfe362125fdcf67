"""Evaluation on the B200 (-m gpu): clm_eval_step against clm_forward and float64 numpy, the same loss as a training
step, the per-read loss on the label-agreement set against the oracle's logits, the forward's status handling, another
pooling mode, and `finetune --val` / `evaluate` end to end.

Tolerances.  `prob` is formed in fp64 from the fp32 logits and rounded once, so it is held to 1e-6 of itself.  The loss is
the training loss's fp32 arithmetic, lse - l_y with lse = max + log(sum): for a confidently right read it is the
difference of two numbers of the logits' size, so its error is a few ulp of the larger of the loss and |logits|, and 1e-6
of that is the bar.  Against the oracle, a logit error e moves lse - l_y by at most 2 e, hence twice the logit tolerance
of tests/test_gpu_labels.py."""

import json
import subprocess
import sys
from dataclasses import replace
from pathlib import Path

import numpy as np
import pytest
import torch

from chimeralm_b200 import synth
from chimeralm_b200 import train as TR
from chimeralm_b200.config import DEFAULT_CONFIG as CFG

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
GOLDEN = ROOT / "tests" / "golden" / "label_agreement.npz"
LOGIT_TOL = 1e-3   # tests/test_gpu_labels.py: default-init head; the probe head's tolerance scales with its gain
HD = "net.head."


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLDEN)


@pytest.fixture(scope="module")
def probe_sd(state_dict, gold):
    """The label-agreement probe head: an output layer fitted on synth's calibration draw, margins of a few units."""
    sd = dict(state_dict)
    sd[HD + "output_layer.weight"] = torch.from_numpy(gold["probe_w"].copy())
    sd[HD + "output_layer.bias"] = torch.from_numpy(gold["probe_b"].copy())
    return sd


def _batch(B, seed, lo=300, hi=1200):
    seqs, cls = synth.label_reads(B, seed, lo, hi)
    return torch.from_numpy(synth.pad_left_ids(seqs)), torch.from_numpy(cls.astype(np.int64))


def _check_rows(logits, targets, loss, prob):
    """loss and prob of eval_step against float64 numpy on the same logits (see the module docstring)."""
    lg = logits.cpu().numpy().astype(np.float64)
    y = targets.cpu().numpy()
    ref_loss = TR.cross_entropy_rows(lg, y)
    ref_prob = 1.0 / (1.0 + np.exp(lg[:, 0] - lg[:, 1]))
    got_loss, got_prob = loss.cpu().numpy().astype(np.float64), prob.cpu().numpy().astype(np.float64)
    scale = np.maximum(ref_loss, np.abs(lg).max(axis=1))
    loss_err = float((np.abs(got_loss - ref_loss) / scale).max())
    prob_err = float((np.abs(got_prob - ref_prob) / ref_prob).max())
    return loss_err, prob_err


@pytest.mark.parametrize("B", [1, 7, 32, 255])
def test_eval_step_matches_forward_and_float64(probe_sd, B):
    from chimeralm_b200.engine import Engine

    ids, y = _batch(B, 700 + B)
    T = ids.shape[1]
    eng = Engine(probe_sd, device=0, max_batch=B, max_tokens=T)
    try:
        ids = ids.to(0)
        f_logits, f_labels = eng.forward(ids, return_labels=True, check=True)
        f_logits, f_labels = f_logits.clone(), f_labels.clone()
        logits, labels, loss, prob = eng.eval_step(ids, y)
    finally:
        eng.close()
    assert torch.equal(logits, f_logits) and torch.equal(labels, f_labels)
    loss_err, prob_err = _check_rows(logits, y, loss, prob)
    print(f"B={B} T={T}: max|logit| {float(logits.abs().max()):.3f}, loss rel err {loss_err:.2e}, prob rel err {prob_err:.2e}")
    assert loss_err <= 1e-6 and prob_err <= 1e-6


def test_eval_loss_is_the_training_loss(state_dict):
    """lr = 0 and dropout = 0: a training step changes nothing and its loss is the mean of eval_step's per-read loss (the
    training step recomputes the classifier on the CUDA cores, the forward's fused head sums in another order)."""
    from chimeralm_b200.engine import Engine

    ids, y = _batch(16, 33, 1000, 3000)
    B, T = ids.shape
    eng = Engine(state_dict, device=0, max_batch=B, max_tokens=T)
    try:
        ids = ids.to(0)
        before = eng.eval_step(ids, y)
        eng.head_train_begin(lr=0.0, weight_decay=0.0, dropout=0.0)
        train_loss = float(eng.head_train_step(ids, y))
        after = eng.eval_step(ids, y)   # between training steps on the same context
        eng.head_train_step(ids, y)
    finally:
        eng.close()
    eval_loss = float(after[2].double().mean())
    print(f"training step loss {train_loss:.8f}, mean eval loss {eval_loss:.8f}")
    assert abs(train_loss - eval_loss) <= 1e-5 * max(1.0, eval_loss)
    assert all(torch.equal(a, b) for a, b in zip(before, after))


def test_eval_on_label_set_against_oracle(probe_sd, gold, state_dict):
    from chimeralm_b200.engine import Engine, pack_reads

    eng = Engine(probe_sd, device=0, max_batch=32, max_tokens=32769)
    loss, labels, targets = [], [], []
    try:
        for seqs, cls in synth.label_eval_batches():
            T = max(len(s) for s in seqs) + 1
            bases, offs = pack_reads([s.tobytes() for s in seqs])
            ids, _ = eng.encode(bases, offs, T, add_cls=False, add_sep=True, pad_left=True, max_bases=32768)
            _, lab, ce, _ = eng.eval_step(ids, torch.from_numpy(cls.astype(np.int64)))
            loss.append(ce.cpu().numpy())
            labels.append(lab.cpu().numpy().astype(np.int64))
            targets.append(cls.astype(np.int64))
        fallbacks = eng.tc_fallbacks
    finally:
        eng.close()
    loss, labels, targets = np.concatenate(loss), np.concatenate(labels), np.concatenate(targets)
    ref_logits = gold["logits_probe"]
    assert len(loss) == len(ref_logits) == int(gold["n_reads"])
    ref_loss = TR.cross_entropy_rows(ref_logits, targets)
    ref_labels = (ref_logits[:, 1] > ref_logits[:, 0]).astype(np.int64)
    gain = float(np.linalg.norm(gold["probe_w"]) / state_dict[HD + "output_layer.weight"].norm())
    tol = 2 * LOGIT_TOL * gain
    err = float(np.abs(loss - ref_loss).max())
    agree = float((labels == ref_labels).mean())
    print(f"{len(loss)} reads: per-read loss max|err| vs oracle {err:.3e} (bar {tol:.3e}), mean loss {loss.mean():.5f} "
          f"(oracle {ref_loss.mean():.5f}), agreement with the oracle's labels {agree:.5f}, fp32 redos {fallbacks}")
    assert err <= tol
    assert agree >= 0.999


def test_eval_status(state_dict):
    from chimeralm_b200.engine import Engine

    eng = Engine(state_dict, device=0, max_batch=2, max_tokens=64)
    try:
        ids = torch.full((2, 64), 8, dtype=torch.uint8)
        ids[1, 5] = 200
        with pytest.raises(IndexError):
            eng.eval_step(ids.to(0), torch.tensor([0, 1]))
        with pytest.raises(ValueError):
            eng.eval_step(torch.full((2, 64), 8, dtype=torch.uint8, device=0), torch.tensor([0, 2]))
    finally:
        eng.close()
    # the input scale of the tensor-core convolution pushed 2^13 too high (the hook of
    # test_gpu_forward.py::test_fp16_range_overflow_switches_to_fp32_conv): the batch is redone on the fp32 convolution
    B, T = 2, 8193
    g = torch.Generator().manual_seed(77)
    ids = torch.randint(7, 11, (B, T), generator=g)
    ids[:, -1] = 1
    ids = ids.to(torch.uint8).cuda()
    y = torch.tensor([1, 0])
    eng = Engine(state_dict, device=0, max_batch=B, max_tokens=T)
    try:
        eng.set_option("tc_conv", 0)
        want = [t.clone() for t in eng.eval_step(ids, y)]
        eng.set_option("tc_conv", 1)
        eng.set_option("tc_scale_shift", 13)
        got = eng.eval_step(ids, y)
        assert eng.tc_fallbacks == 1
        assert all(torch.equal(a, b) for a, b in zip(got, want))
    finally:
        eng.close()


def test_eval_mean_pooling(state_dict):
    from chimeralm_b200.engine import Engine

    sd_mean = {k: v for k, v in state_dict.items() if ".attention." not in k}
    ids, y = _batch(5, 91)
    eng = Engine(sd_mean, device=0, cfg=replace(CFG, pooling_type="mean"), max_batch=5, max_tokens=ids.shape[1])
    try:
        ids = ids.to(0)
        f_logits = eng.forward(ids, check=True).clone()
        logits, labels, loss, prob = eng.eval_step(ids, y)
    finally:
        eng.close()
    assert torch.equal(logits, f_logits)
    loss_err, prob_err = _check_rows(logits, y, loss, prob)
    assert loss_err <= 1e-6 and prob_err <= 1e-6


def _write_fq(path, batches):
    n = 0
    with path.open("w") as f:
        for seqs, cls in batches:
            for s, c in zip(seqs, cls):
                f.write(f"@read{n}|{int(c)}\n{s.tobytes().decode()}\n+\n{'I' * len(s)}\n")
                n += 1
    return n


def _cli(*args):
    r = subprocess.run([sys.executable, "-m", "chimeralm_b200", *map(str, args)], cwd=ROOT, capture_output=True, text=True)
    print(r.stdout[-2000:], r.stderr[-3000:])
    assert r.returncode == 0
    return r


def test_finetune_val_then_evaluate_cli(tmp_path):
    """Seeded random-init model; the head is trained on synth's calibration draw and validated on the label-agreement
    evaluation reads.  The checkpoint is the chosen epoch's: `evaluate` reproduces that epoch's validation metrics
    exactly (same batches, same kernels)."""
    train_fq, val_fq = tmp_path / "train.fq", tmp_path / "val.fq"
    _write_fq(train_fq, synth.label_calibration_batches())
    n_val = _write_fq(val_fq, synth.label_eval_batches())
    out = tmp_path / "tuned.ckpt"
    _cli("finetune", train_fq, "-o", out, "--val", val_fq, "--epochs", 4, "--lr", "1e-3", "--batch-size", 32, "--seed", 0)
    rep = json.loads(Path(str(out) + ".val.json").read_text())
    recs = rep["epochs"]
    assert [r["epoch"] for r in recs] == [0, 1, 2, 3, 4] and recs[0]["train_loss"] is None
    assert rep["best_epoch"] == TR.best_epoch(recs) >= 1 and not rep["stopped_early"]
    best = recs[rep["best_epoch"]]
    m1, m2 = tmp_path / "m1.json", tmp_path / "m2.json"
    per_read = tmp_path / "reads.tsv"
    _cli("evaluate", val_fq, "--ckpt", out, "-o", m1, "--per-read", per_read)
    _cli("evaluate", val_fq, "--ckpt", out, "-o", m2)
    got = json.loads(m1.read_text())
    print(f"chosen epoch {rep['best_epoch']}: " + json.dumps(best))
    assert got == {k: v for k, v in best.items() if k not in ("epoch", "train_loss")}
    assert m1.read_bytes() == m2.read_bytes()
    assert got["reads"] == n_val and got["accuracy"] >= 0.95
    lines = per_read.read_text().splitlines()
    assert lines[0].split("\t") == ["name", "target", "label", "p_chimera", "loss"] and len(lines) == n_val + 1
    rows = [ln.split("\t") for ln in lines[1:]]
    assert [r[0] for r in rows] == [f"read{i}|{r[1]}" for i, r in enumerate(rows)]   # input order
    acc = np.mean([r[1] == r[2] for r in rows])
    assert acc == got["accuracy"]
    assert abs(np.mean([float(r[4]) for r in rows]) - got["loss"]) <= 1e-6 * max(1.0, got["loss"])
