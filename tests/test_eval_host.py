"""Host side of evaluation (no GPU): the metrics against hand-worked cases and a brute-force AUROC, the float64
cross-entropy mirror, the choice of the epoch to keep and early stopping, and the `evaluate` command's input checks."""

import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from chimeralm_b200 import train as TR

ROOT = Path(__file__).resolve().parents[1]


def _metrics(y, yhat, prob=None, loss=None):
    y = np.asarray(y)
    prob = np.asarray(yhat, np.float64) if prob is None else prob
    loss = np.zeros(len(y)) if loss is None else loss
    return TR.binary_metrics(y, yhat, prob, loss)


def test_all_correct():
    m = _metrics([0, 1, 1, 0, 1], [0, 1, 1, 0, 1], prob=[0.1, 0.9, 0.8, 0.3, 0.7], loss=[0.1, 0.2, 0.3, 0.4, 0.5])
    assert m["accuracy"] == 1.0 and m["precision"] == 1.0 and m["recall"] == 1.0 and m["f1"] == 1.0
    assert m["auroc"] == 1.0
    assert m["confusion"] == [[2, 0], [0, 3]]
    assert m["reads"] == 5 and m["loss"] == pytest.approx(0.3, abs=1e-15)


def test_all_wrong():
    m = _metrics([0, 1, 1, 0], [1, 0, 0, 1], prob=[0.9, 0.2, 0.1, 0.8])
    assert m["accuracy"] == 0.0 and m["precision"] == 0.0 and m["recall"] == 0.0 and m["f1"] == 0.0
    assert m["auroc"] == 0.0
    assert m["confusion"] == [[0, 2], [2, 0]]


def test_no_predicted_positives():
    # tp + fp = 0: precision is 0 (torchmetrics' zero_division default), recall and F1 are 0 as tp = 0
    m = _metrics([0, 1, 0, 1, 0], [0, 0, 0, 0, 0], prob=[0.1, 0.4, 0.2, 0.3, 0.05])
    assert m["precision"] == 0.0 and m["recall"] == 0.0 and m["f1"] == 0.0
    assert m["accuracy"] == pytest.approx(0.6, abs=1e-15)
    assert m["confusion"] == [[3, 0], [2, 0]]
    assert m["auroc"] == 1.0   # the ranking is perfect although no read crosses the decision threshold


def test_one_class_only():
    m = _metrics([1, 1, 1], [1, 0, 1], prob=[0.9, 0.4, 0.6])
    assert m["auroc"] is None
    assert m["precision"] == 1.0 and m["recall"] == pytest.approx(2 / 3, abs=1e-15)
    assert m["f1"] == pytest.approx(0.8, abs=1e-15)   # 2 tp / (2 tp + fp + fn) = 4 / 5
    assert m["confusion"] == [[0, 0], [1, 2]]
    assert _metrics([0, 0], [0, 0], prob=[0.1, 0.2])["auroc"] is None


def test_tied_probabilities():
    # positives at 0.5, 0.5, 0.9; negatives at 0.5, 0.1.  Pairs (pos, neg): (0.5, 0.5) = 1/2 twice, (0.9, 0.5) = 1,
    # every positive over 0.1 = 3: (2 * 0.5 + 1 + 3) / 6 = 5 / 6
    m = _metrics([1, 1, 1, 0, 0], [1, 1, 1, 1, 0], prob=[0.5, 0.5, 0.9, 0.5, 0.1])
    assert m["auroc"] == pytest.approx(5 / 6, abs=1e-15)
    assert _metrics([0, 1, 0, 1], [0, 0, 0, 0], prob=[0.3] * 4)["auroc"] == 0.5   # all tied: chance


def test_auroc_against_pair_count():
    rng = np.random.default_rng(5)
    for trial in range(20):
        n = int(rng.integers(2, 300))
        y = rng.integers(0, 2, n)
        y[0], y[-1] = 0, 1
        prob = rng.integers(0, 12, n) / 11.0   # few distinct values: many ties
        pos, neg = prob[y == 1], prob[y == 0]
        d = pos[:, None] - neg[None, :]
        want = ((d > 0).sum() + 0.5 * (d == 0).sum()) / d.size
        assert TR.auroc(y, prob) == pytest.approx(want, abs=1e-12), trial


def test_metrics_reject_mismatched_lengths():
    with pytest.raises(ValueError):
        TR.binary_metrics([0, 1], [0], [0.1, 0.2], [0.0, 0.0])
    with pytest.raises(ValueError):
        TR.binary_metrics([], [], [], [])


def test_cross_entropy_mirror():
    lg = np.array([[1e4, -1e4], [-1e4, 1e4], [1e4, 1e4], [0.5, -0.25], [-3.0, 2.0]], np.float32)
    y = np.array([0, 0, 1, 1, 1])
    ce = TR.cross_entropy_rows(lg, y)
    assert np.all(np.isfinite(ce))
    assert ce[0] == 0.0 and ce[1] == 2e4 and ce[2] == pytest.approx(np.log(2.0), rel=1e-15)
    d = lg[3:].astype(np.float64)
    softplus = np.log1p(np.exp(d[:, 0] - d[:, 1]))   # -log softmax_1, the other closed form
    assert np.allclose(ce[3:], softplus, rtol=1e-12, atol=0)


def _recs(rows):
    return [{"epoch": e, "f1": f1, "loss": loss} for e, f1, loss in rows]


def test_best_epoch_rule():
    # epoch 0 (before training) is never chosen, even when it is the best
    assert TR.best_epoch(_recs([(0, 0.99, 0.01), (1, 0.5, 0.7), (2, 0.6, 0.9)])) == 2
    # equal F1: the lower loss wins
    assert TR.best_epoch(_recs([(0, 0.0, 1.0), (1, 0.8, 0.5), (2, 0.8, 0.4), (3, 0.7, 0.1)])) == 2
    # equal F1 and loss: the earlier epoch
    assert TR.best_epoch(_recs([(0, 0.0, 1.0), (1, 0.8, 0.4), (2, 0.8, 0.4), (3, 0.8, 0.4)])) == 1
    assert TR.best_epoch(_recs([(0, 0.3, 1.0)])) == 0


def test_patience_counts_epochs_without_a_better_f1():
    assert TR.epochs_without_improvement(_recs([(0, 0.9, 0.1)])) == 0
    assert TR.epochs_without_improvement(_recs([(0, 0.9, 0.1), (1, 0.2, 0.9)])) == 0   # epoch 0 sets no bar
    rows = [(0, 0.0, 1.0), (1, 0.5, 0.9), (2, 0.7, 0.8), (3, 0.7, 0.1), (4, 0.6, 0.2)]
    # an equal F1 is not a better one, even at a lower loss
    assert [TR.epochs_without_improvement(_recs(rows[:k])) for k in range(2, 6)] == [0, 0, 1, 2]
    assert TR.epochs_without_improvement(_recs(rows + [(5, 0.71, 0.5)])) == 0


def test_evaluate_help():
    r = subprocess.run([sys.executable, "-m", "chimeralm_b200", "evaluate", "--help"], cwd=ROOT, capture_output=True,
                       text=True)
    assert r.returncode == 0
    for flag in ("--ckpt", "--batch-size", "--output", "--per-read"):
        assert flag in r.stdout


def test_evaluate_rejects_unlabelled_reads(tmp_path):
    fq = tmp_path / "u.fq"
    fq.write_text("@a|0\nACGT\n+\nIIII\n@b\nACGA\n+\nIIII\n")
    r = subprocess.run([sys.executable, "-m", "chimeralm_b200", "evaluate", str(fq), "--ckpt", str(tmp_path / "m.ckpt")],
                       cwd=ROOT, capture_output=True, text=True)
    assert r.returncode != 0
    assert "read 'b' has no 0/1 label" in r.stdout + r.stderr


def test_finetune_patience_needs_validation(tmp_path):
    with pytest.raises(ValueError, match="patience"):
        TR.finetune(tmp_path / "t.fq", None, tmp_path / "o.ckpt", patience=2)
