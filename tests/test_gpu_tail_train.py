"""Training the last block's tail (out_proj, norm2, fc1, fc2) and ln_f together with the head on the B200 (-m gpu):
gradients against fp64 autograd on the forward's own block input r0 and conv output y, the head's gradients and the
determinism of the tail's, the AdamW step, the refreshed forward against a freshly built engine, the frozen rest of the
backbone, the bad-status rule, learning through the CLI, and the rejected calls.

Gradient bound: 3e-2 relative L2 per tail tensor, the scorer's bound (tests/test_gpu_head_train.py), for the same reason:
the backward multiplies bf16 operands (dz, dr2, dh, dr1, the recomputed activations) on the tensor cores.  The bound is a
target, not a measurement; each case prints its figures."""

import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from chimeralm_b200.config import DEFAULT_CONFIG as CFG

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
TAIL_TOL = 3e-2
LOSS_TOL = 1e-3
LOGIT_TOL = 1e-3
P = 0.1
D = CFG.d_model
HD = "net.head."
HEAD_NAMES = ["attention.0.weight", "attention.0.bias", "attention.2.weight", "attention.2.bias", "classifier.0.weight",
              "classifier.0.bias", "classifier.3.weight", "classifier.3.bias", "classifier.6.layers.0.weight",
              "classifier.6.layers.0.bias", "classifier.6.layers.3.weight", "classifier.6.layers.3.bias",
              "output_layer.weight", "output_layer.bias"]


def _tail():
    from chimeralm_b200.engine import tail_keys

    return tail_keys(CFG.n_layer)


def _label_batch(B, lo, hi, seed):
    from chimeralm_b200 import synth

    seqs, cls = synth.label_reads(B, seed, lo, hi)
    return torch.from_numpy(synth.pad_left_ids(seqs)), torch.from_numpy(cls.astype(np.int64))


def _k2_batch(B=8):
    g = torch.Generator().manual_seed(11)
    ids = torch.randint(7, 11, (B, 8193), generator=g, dtype=torch.int64)
    ids[:, -1] = 1
    return ids.to(torch.uint8), torch.arange(B) % 2


def _long_batch():
    g = torch.Generator().manual_seed(12)
    ids = torch.randint(7, 11, (2, 32769), generator=g, dtype=torch.int64)
    ids[:, -1] = 1
    ids[1, :12001] = 4   # a 20 768-token read left-padded to the batch
    return ids.to(torch.uint8), torch.tensor([1, 0])


def _r0_y(eng, B, T):
    """Block L's input residual r0 and conv output y of the last forward, [B, T, 256] fp32."""
    from chimeralm_b200.engine import r32_to_rows

    M = B * T
    r0 = r32_to_rows(eng.debug_copy("resid", ((M + 31) // 32 * 32 * D,), torch.float32), M).reshape(B, T, D)
    Tp = (T + 127) // 128 * 128
    y = eng.debug_copy("y", (B, D, Tp), torch.bfloat16)[:, :, :T].transpose(1, 2).float()
    return r0.clone(), y.contiguous()


def _ref(sd, r0, y, targets, masks, p):
    """fp64 autograd through the tail, ln_f and the head (dropout keep-masks [3, B, 512] at classifier.2 / .5 /
    .6.layers.2) on the given r0 and y.  Returns (loss, {key: grad})."""
    dev, dd = r0.device, torch.float64
    keys = _tail() + [HD + n for n in HEAD_NAMES]
    w = {k: sd[k].to(dev, dd).clone().requires_grad_(True) for k in keys}
    tk = _tail()
    eps = CFG.layer_norm_epsilon
    r1 = r0.to(dd) + F.linear(y.to(dd), w[tk[0]], w[tk[1]])
    x2 = F.layer_norm(r1, (D,), w[tk[2]], w[tk[3]], eps)
    a = F.gelu(F.linear(x2, w[tk[4]], w[tk[5]]), approximate="tanh")
    r2 = r1 + F.linear(a, w[tk[6]], w[tk[7]])
    hid = F.layer_norm(r2, (D,), w[tk[8]], w[tk[9]], eps)
    m = torch.from_numpy(masks).to(dev, dd) * float(np.float32(1.0 / (1.0 - p))) if p > 0 else None

    def drop(x, i):
        return x if m is None else x * m[i]

    s = F.linear(F.gelu(F.linear(hid, w[HD + "attention.0.weight"], w[HD + "attention.0.bias"])),
                 w[HD + "attention.2.weight"], w[HD + "attention.2.bias"])
    pooled = (hid * torch.softmax(s, dim=1)).sum(dim=1)
    x = drop(F.gelu(F.linear(pooled, w[HD + "classifier.0.weight"], w[HD + "classifier.0.bias"])), 0)
    x = drop(F.gelu(F.linear(x, w[HD + "classifier.3.weight"], w[HD + "classifier.3.bias"])), 1)
    r = drop(F.gelu(F.linear(x, w[HD + "classifier.6.layers.0.weight"], w[HD + "classifier.6.layers.0.bias"])), 2)
    x = F.linear(r, w[HD + "classifier.6.layers.3.weight"], w[HD + "classifier.6.layers.3.bias"]) + x
    logits = F.linear(x, w[HD + "output_layer.weight"], w[HD + "output_layer.bias"])
    loss = F.cross_entropy(logits, targets.to(dev))
    loss.backward()
    return float(loss), {k: w[k].grad.float().cpu() for k in keys}


def _engine(sd, ids, tail_lr=0.0, **hp):
    from chimeralm_b200.engine import Engine

    B, T = ids.shape
    eng = Engine(sd, device=0, max_batch=B, max_tokens=T)
    eng.head_train_begin(**{"lr": 0.0, "weight_decay": 0.0, "dropout": P, "seed": 1234, **hp})
    if tail_lr is not None:
        eng.tail_train_begin(tail_lr)
    return eng


@pytest.mark.parametrize("case", ["k2", "padded_1_4kb", "long_2x32769"])
def test_tail_gradient_parity_with_autograd(state_dict, case):
    from chimeralm_b200 import train as TR

    ids, y = {"k2": _k2_batch, "long_2x32769": _long_batch}.get(case, lambda: _label_batch(16, 1000, 4000, 31))()
    B, T = ids.shape
    eng = _engine(state_dict, ids)
    try:
        loss = float(eng.head_train_step(ids.to(0), y))
        got = {k: eng.head_grad(k).cpu() for k in _tail()}
        r0, yy = _r0_y(eng, B, T)
    finally:
        eng.close()
    ref_loss, ref = _ref(state_dict, r0, yy, y, TR.dropout_masks(1234, 0, B, P), P)
    errs = {k.rsplit("backbone.", 1)[1]: float((got[k] - ref[k]).norm() / ref[k].norm()) for k in _tail()}
    print(f"{case} {B}x{T}: loss {loss:.6f} (autograd {ref_loss:.6f}); rel L2 tail grad errors "
          + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert abs(loss - ref_loss) <= LOSS_TOL * max(1.0, ref_loss)
    bad = {k: v for k, v in errs.items() if not v <= TAIL_TOL}
    assert not bad, bad


def test_head_grads_unchanged_and_tail_grads_deterministic(state_dict):
    """With the tail on, the head's 14 gradients are bit-identical to a head-only step; two fresh engines taking the
    same step give bit-identical tail gradients."""
    ids, y = _label_batch(12, 1000, 3000, 33)
    grads = []
    for tail_lr in (None, 1e-3, 1e-3):
        eng = _engine(state_dict, ids, tail_lr=tail_lr, lr=1e-3)
        try:
            eng.head_train_step(ids.to(0), y)
            g = {HD + n: eng.head_grad(HD + n).cpu() for n in HEAD_NAMES}
            if tail_lr is not None:
                g.update({k: eng.head_grad(k).cpu() for k in _tail()})
            grads.append(g)
        finally:
            eng.close()
    head_only, a, b = grads
    assert all(torch.equal(head_only[k], a[k]) for k in head_only)
    assert all(torch.equal(a[k], b[k]) for k in a)
    assert all(float(a[k].abs().max()) > 0 for k in _tail())


def test_tail_step_matches_torch_adamw(state_dict):
    ids, y = _label_batch(6, 1000, 2500, 41)
    hp = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.05)
    tail_lr = 2e-3
    eng = _engine(state_dict, ids, tail_lr=tail_lr, **hp)
    try:
        eng.head_train_step(ids.to(0), y)
        grads = {k: eng.head_grad(k).cpu() for k in _tail()}
        got = eng.tail_state_dict()
    finally:
        eng.close()
    params = {k: torch.nn.Parameter(state_dict[k].clone()) for k in _tail()}
    opt = torch.optim.AdamW(list(params.values()), foreach=False, **{**hp, "lr": tail_lr})
    for k, prm in params.items():
        prm.grad = grads[k].clone()
    opt.step()
    for k in _tail():
        ref = params[k].detach()
        assert float((got[k] - ref).norm()) <= 1e-6 * float(ref.norm()), k
        assert not torch.equal(got[k], state_dict[k]), k


def test_refreshed_forward_equals_a_fresh_engine(state_dict):
    """After 5 steps the training engine's forward equals, bit for bit, that of an engine built from the exported
    weights, on a tensor-core-conv batch and an fp32-conv batch, with another model's forward on the same device in
    between (the block-tail constant bank is per device).  The unfused forward agrees within the logit bar."""
    from chimeralm_b200 import train as TR
    from chimeralm_b200.engine import Engine
    from chimeralm_b200.weights import make_state_dict

    train_ids, train_y = _label_batch(8, 1000, 2000, 43)
    k2, _ = _k2_batch(4)
    short, _ = _label_batch(8, 1000, 2000, 44)
    eng = _engine(state_dict, train_ids, tail_lr=1e-3, lr=1e-3, weight_decay=0.01)
    other = Engine(make_state_dict(3), device=0, max_batch=4, max_tokens=8193)
    try:
        for _ in range(5):
            eng.head_train_step(train_ids.to(0), train_y)
        tuned = TR.tuned_state_dict(state_dict, eng, train_tail=True)
        other.forward(k2.to(0), check=True)
        outs = [eng.forward(x.to(0), return_labels=True, check=True) for x in (k2, short)]
        eng.set_option("fused_mlp", 0)
        unfused = [eng.forward(x.to(0), check=True) for x in (k2, short)]
        eng.set_option("fused_mlp", 1)
    finally:
        eng.close()
        other.close()
    fresh = Engine(tuned, device=0, max_batch=8, max_tokens=8193, token_budget=4 * 8193)
    try:
        ref = [fresh.forward(x.to(0), return_labels=True, check=True) for x in (k2, short)]
    finally:
        fresh.close()
    for (lg, lb), (rl, rb), uf in zip(outs, ref, unfused):
        scale = max(1.0, float(rl.abs().max()))
        print(f"refreshed vs fresh: max|diff| {float((lg - rl).abs().max()):.3e}; unfused {float((uf - lg).abs().max()):.3e}")
        assert torch.equal(lg.cpu(), rl.cpu()) and torch.equal(lb.cpu(), rb.cpu())
        assert float((uf - lg).abs().max()) <= LOGIT_TOL * scale
    for k in _tail():
        assert not torch.equal(tuned[k], state_dict[k]), k


def test_frozen_backbone_after_20_steps(state_dict):
    """After 20 steps with the tail on: the filters of every layer, block L's input residual r0 and its conv output y
    are bit-identical, every tensor outside the 24 trained ones is the input's, and the loss fell."""
    from chimeralm_b200 import train as TR
    from chimeralm_b200.engine import Engine

    ids, y = _label_batch(8, 1000, 3000, 51)
    B, T = ids.shape
    ref = Engine(state_dict, device=0, max_batch=B, max_tokens=T)
    try:
        ref.forward(ids.to(0), check=True)
        r0a, ya = _r0_y(ref, B, T)
        filt0 = [ref.get_filter(l, T).cpu() for l in range(CFG.n_layer)]
    finally:
        ref.close()
    eng = _engine(state_dict, ids, tail_lr=1e-3, lr=1e-3, weight_decay=0.01)
    try:
        losses = [float(eng.head_train_step(ids.to(0), y)) for _ in range(20)]
        eng.forward(ids.to(0), check=True)
        r0b, yb = _r0_y(eng, B, T)
        filt1 = [eng.get_filter(l, T).cpu() for l in range(CFG.n_layer)]
        tuned = TR.tuned_state_dict(state_dict, eng, train_tail=True)
    finally:
        eng.close()
    print(f"20 steps with the tail on one batch: loss {losses[0]:.4f} -> {losses[-1]:.4f}")
    assert torch.equal(r0a.cpu(), r0b.cpu()) and torch.equal(ya.cpu(), yb.cpu())
    assert all(torch.equal(a, b) for a, b in zip(filt0, filt1))
    trained = set(_tail()) | {HD + n for n in HEAD_NAMES}
    assert len(trained) == 24
    assert all(torch.equal(tuned[k], state_dict[k]) for k in state_dict if k not in trained)
    assert losses[-1] < losses[0]


def test_bad_status_changes_nothing(state_dict):
    ids = torch.full((2, 64), 8, dtype=torch.uint8)
    ids[1, 5] = 200
    eng = _engine(state_dict, ids, tail_lr=1e-2, lr=1e-2)
    try:
        before = {**eng.head_state_dict(), **eng.tail_state_dict()}
        with pytest.raises(IndexError):
            eng.head_train_step(ids.to(0), torch.tensor([0, 1]))
        after = {**eng.head_state_dict(), **eng.tail_state_dict()}
    finally:
        eng.close()
    assert all(torch.equal(before[k], after[k]) for k in before)


def test_rejected_calls(state_dict):
    from chimeralm_b200 import _lib
    from chimeralm_b200.engine import Engine

    ids, y = _label_batch(2, 300, 600, 61)
    eng = Engine(state_dict, device=0, max_batch=2, max_tokens=ids.shape[1])
    try:
        with pytest.raises(_lib.ChimeraLMNativeError, match="before clm_head_train_begin"):
            eng.tail_train_begin(1e-3)
        eng.head_train_begin(lr=1e-3)
        with pytest.raises(_lib.ChimeraLMNativeError, match="before clm_tail_train_begin"):
            eng.head_grad(_tail()[0])
        eng.tail_train_begin(1e-3)
        with pytest.raises(_lib.ChimeraLMNativeError, match="already in training"):
            eng.tail_train_begin(1e-3)
        eng.set_option("skip_dead_res", 0)
        with pytest.raises(_lib.ChimeraLMNativeError, match="skip_dead_res"):
            eng.head_train_step(ids.to(0), y)
        eng.set_option("skip_dead_res", 1)
        eng.head_train_step(ids.to(0), y)
    finally:
        eng.close()
    eng = Engine(state_dict, device=0, max_batch=2, max_tokens=ids.shape[1])
    try:
        eng.head_train_begin(lr=1e-3)
        eng.head_train_step(ids.to(0), y)
        with pytest.raises(_lib.ChimeraLMNativeError, match="after a clm_head_train_step"):
            eng.tail_train_begin(1e-3)
        assert torch.equal(eng.head_export(_tail()[0]), state_dict[_tail()[0]])   # not in training: the loaded value
    finally:
        eng.close()


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


def test_finetune_train_tail_val_then_evaluate_cli(tmp_path):
    """`finetune --train-tail --val` on synth's composition classes reaches the head-only bar on the held-out reads, and
    `evaluate` on the saved checkpoint reproduces the chosen epoch's validation record exactly."""
    from chimeralm_b200 import synth
    from chimeralm_b200 import train as TR
    from chimeralm_b200.weights import load_checkpoint, make_state_dict

    train_fq, val_fq = tmp_path / "train.fq", tmp_path / "val.fq"
    _write_fq(train_fq, synth.label_calibration_batches())
    n_val = _write_fq(val_fq, synth.label_eval_batches())
    out = tmp_path / "tuned.ckpt"
    _cli("finetune", train_fq, "-o", out, "--val", val_fq, "--epochs", 4, "--lr", "1e-3", "--batch-size", 32, "--seed", 0,
         "--train-tail", "--tail-lr", "3e-4")
    rep = json.loads(Path(str(out) + ".val.json").read_text())
    best = rep["epochs"][rep["best_epoch"]]
    assert rep["best_epoch"] == TR.best_epoch(rep["epochs"]) >= 1
    m1 = tmp_path / "m1.json"
    _cli("evaluate", val_fq, "--ckpt", out, "-o", m1)
    got = json.loads(m1.read_text())
    print(f"chosen epoch {rep['best_epoch']}: " + json.dumps(best))
    assert got == {k: v for k, v in best.items() if k not in ("epoch", "train_loss")}
    assert got["reads"] == n_val and got["accuracy"] >= 0.95
    tuned, base = load_checkpoint(out), make_state_dict(0)
    trained = set(_tail()) | {HD + n for n in HEAD_NAMES}
    assert list(tuned) == list(base)
    assert all(torch.equal(tuned[k], base[k]) for k in base if k not in trained)
    assert all(not torch.equal(tuned[k], base[k]) for k in _tail())
