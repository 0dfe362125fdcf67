"""Head fine-tuning on the B200 (-m gpu): gradients against torch autograd through the oracle's head, the AdamW step
against torch.optim.AdamW, the forward after a step against the oracle, the frozen backbone, learning on labelled
composition classes and the rejected inputs.

Gradient bounds, per-tensor relative L2 error against autograd on the oracle's fp32 hidden states:
  classifier tensors <= 2e-2 (fp32 arithmetic on the forward's pooled vector; measured on one B200: <= 3.7e-3);
  scorer tensors (attention.*) <= 3e-2.  They multiply bf16 operands (the rows XN the forward wrote, dz rounded to bf16 for
  the tensor cores, ~4e-3 relative per element), and ds_t = w_t (h_t - pooled) . dp is a difference of nearly equal terms
  that amplifies the rounding of h_t.  Measured on one B200: 6e-3 at 2 x 32 769 tokens, 1.7e-2 at 8 x 8 193, 2.4e-2 on 16
  heavily left-padded reads of 1-4 kb (the case with the fewest tokens per read).  Each case prints its figures."""

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
GRAD_TOL = 2e-2          # classifier tensors
SCORER_GRAD_TOL = 3e-2   # attention.* (bf16 operands, see above)
LOGIT_TOL = 1e-3
P = 0.1
HEAD_NAMES = ["attention.0.weight", "attention.0.bias", "attention.2.weight", "attention.2.bias", "classifier.0.weight",
              "classifier.0.bias", "classifier.3.weight", "classifier.3.bias", "classifier.6.layers.0.weight",
              "classifier.6.layers.0.bias", "classifier.6.layers.3.weight", "classifier.6.layers.3.bias",
              "output_layer.weight", "output_layer.bias"]


def _hidden(sd, ids):
    """The oracle's fp32 hidden states (ln_f output) as an ordinary tensor."""
    from oracle import hyena_oracle as O

    with torch.inference_mode():
        _, h = O.forward(sd, ids, CFG, return_hidden=True)
    return h.clone()


def _ref_grads(sd, hidden, targets, masks, p):
    """torch autograd of mean cross-entropy through the head with the given dropout keep-masks [3, B, 512].  With p = 0
    the forward IS oracle.hyena_oracle.head; otherwise the same lines with the masks applied at classifier.2,
    classifier.5 and classifier.6.layers.2."""
    from oracle import hyena_oracle as O

    params = {O.HD + n: sd[O.HD + n].clone().requires_grad_(True) for n in HEAD_NAMES}
    w = dict(sd)
    w.update(params)
    if p == 0:
        logits = O.head(w, hidden)
    else:
        m = torch.from_numpy(masks).float() * float(np.float32(1.0 / (1.0 - p)))
        a = F.gelu(F.linear(hidden, w[O.HD + "attention.0.weight"], w[O.HD + "attention.0.bias"]))
        s = F.linear(a, w[O.HD + "attention.2.weight"], w[O.HD + "attention.2.bias"])
        pooled = (hidden * torch.softmax(s, dim=1)).sum(dim=1)
        x = F.gelu(F.linear(pooled, w[O.HD + "classifier.0.weight"], w[O.HD + "classifier.0.bias"])) * m[0]
        x = F.gelu(F.linear(x, w[O.HD + "classifier.3.weight"], w[O.HD + "classifier.3.bias"])) * m[1]
        r = F.gelu(F.linear(x, w[O.HD + "classifier.6.layers.0.weight"], w[O.HD + "classifier.6.layers.0.bias"])) * m[2]
        x = F.linear(r, w[O.HD + "classifier.6.layers.3.weight"], w[O.HD + "classifier.6.layers.3.bias"]) + x
        logits = F.linear(x, w[O.HD + "output_layer.weight"], w[O.HD + "output_layer.bias"])
    loss = F.cross_entropy(logits, targets)
    loss.backward()
    return float(loss), {n: params[O.HD + n].grad for n in HEAD_NAMES}


def _label_batch(B, lo, hi, seed):
    from chimeralm_b200 import synth

    seqs, cls = synth.label_reads(B, seed, lo, hi)
    return torch.from_numpy(synth.pad_left_ids(seqs)), torch.from_numpy(cls.astype(np.int64))


def _k2_batch():
    g = torch.Generator().manual_seed(11)
    ids = torch.randint(7, 11, (8, 8193), generator=g, dtype=torch.int64)
    ids[:, -1] = 1
    return ids.to(torch.uint8), torch.tensor([0, 1, 1, 0, 1, 0, 0, 1])


def _long_batch():
    g = torch.Generator().manual_seed(12)
    ids = torch.randint(7, 11, (2, 32769), generator=g, dtype=torch.int64)
    ids[:, -1] = 1
    ids[1, :12001] = 4   # a 20 768-token read left-padded to the batch
    return ids.to(torch.uint8), torch.tensor([1, 0])


@pytest.mark.parametrize("case,p", [("k2", P), ("padded_1_4kb", P), ("long_2x32769", P), ("padded_1_4kb", 0.0)])
def test_gradient_parity_with_autograd(state_dict, case, p):
    from chimeralm_b200 import train as TR
    from chimeralm_b200.engine import Engine

    if case == "k2":
        ids, y = _k2_batch()
    elif case == "long_2x32769":
        ids, y = _long_batch()
    else:
        ids, y = _label_batch(16, 1000, 4000, 31)
    B, T = ids.shape
    eng = Engine(state_dict, device=0, max_batch=B, max_tokens=T)
    try:
        eng.head_train_begin(lr=0.0, weight_decay=0.0, dropout=p, seed=1234)
        loss = eng.head_train_step(ids.to(0), y)
        got = {n: eng.head_grad(n).cpu() for n in HEAD_NAMES}
    finally:
        eng.close()
    masks = TR.dropout_masks(1234, 0, B, p)
    ref_loss, ref = _ref_grads(state_dict, _hidden(state_dict, ids.long()), y, masks, p)
    errs = {}
    for n in HEAD_NAMES:
        if n == "attention.2.bias":   # sum_t ds_t = 0 exactly: compare with the scale of the attention.2.weight gradient
            assert abs(float(got[n]) - float(ref[n])) <= 1e-3 * float(ref["attention.2.weight"].norm()), (got[n], ref[n])
            continue
        errs[n] = float((got[n] - ref[n]).norm() / ref[n].norm())
    print(f"{case} {B}x{T} p={p}: loss {float(loss):.6f} (autograd {ref_loss:.6f}); rel L2 grad errors "
          + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert abs(float(loss) - ref_loss) <= 1e-3 * max(1.0, ref_loss)
    bad = {k: v for k, v in errs.items() if not v <= (SCORER_GRAD_TOL if k.startswith("attention.") else GRAD_TOL)}
    assert not bad, bad


def test_step_parity_with_torch_adamw_and_refreshed_forward(state_dict):
    """One step: the exported head equals torch.optim.AdamW applied to the GPU's own gradients; the forward then reads
    the updated head (logits against the oracle with those weights, within the logit bar scaled to the logits' size: a
    step of this size grows them)."""
    from oracle import hyena_oracle as O

    from chimeralm_b200.engine import Engine

    ids, y = _label_batch(6, 1000, 2500, 41)
    B, T = ids.shape
    hp = dict(lr=2e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.05)
    eng = Engine(state_dict, device=0, max_batch=B, max_tokens=T)
    try:
        before = eng.forward(ids.to(0), check=True).cpu()
        eng.head_train_begin(dropout=P, seed=5, **hp)
        eng.head_train_step(ids.to(0), y)
        grads = {n: eng.head_grad(n).cpu() for n in HEAD_NAMES}
        got = {n: eng.head_export(n) for n in HEAD_NAMES}
        logits = eng.forward(ids.to(0), check=True).cpu()
    finally:
        eng.close()
    params = {n: torch.nn.Parameter(state_dict[O.HD + n].clone()) for n in HEAD_NAMES}
    opt = torch.optim.AdamW(list(params.values()), foreach=False, **hp)
    for n, prm in params.items():
        prm.grad = grads[n].clone()
    opt.step()
    for n in HEAD_NAMES:
        ref = params[n].detach()
        assert float((got[n] - ref).norm()) <= 1e-6 * float(ref.norm()), n
        assert not torch.equal(got[n], state_dict[O.HD + n]), n   # the step moved every tensor
    tuned = dict(state_dict)
    tuned.update({O.HD + n: got[n] for n in HEAD_NAMES})
    ref_logits = O.forward(tuned, ids.long(), CFG)
    err = float((logits - ref_logits).abs().max())
    scale = max(1.0, float(ref_logits.abs().max()))
    moved = float((logits - before).abs().max())
    print(f"refreshed forward: logits max|err| vs oracle with the updated head {err:.3e} (max|logit| {scale:.3f}); "
          f"the step moved the logits by up to {moved:.3e}")
    assert err <= LOGIT_TOL * scale
    assert moved >= 20 * LOGIT_TOL * scale


def test_backbone_untouched_after_20_steps(state_dict):
    from chimeralm_b200.engine import Engine

    ids, y = _label_batch(8, 1000, 3000, 51)
    B, T = ids.shape
    eng = Engine(state_dict, device=0, max_batch=B, max_tokens=T)
    try:
        n_xn = B * T * CFG.d_model
        eng.forward(ids.to(0), check=True)
        xn0 = eng.debug_copy("xn", (n_xn,), torch.bfloat16).cpu()
        filt0 = [eng.get_filter(l, T).cpu() for l in range(CFG.n_layer)]
        eng.head_train_begin(lr=1e-3, dropout=P, seed=9)
        losses = [float(eng.head_train_step(ids.to(0), y)) for _ in range(20)]
        eng.forward(ids.to(0), check=True)
        xn1 = eng.debug_copy("xn", (n_xn,), torch.bfloat16).cpu()
        filt1 = [eng.get_filter(l, T).cpu() for l in range(CFG.n_layer)]
        head = eng.head_state_dict()
    finally:
        eng.close()
    print(f"20 steps on one batch: loss {losses[0]:.4f} -> {losses[-1]:.4f}")
    assert torch.equal(xn0, xn1)
    assert all(torch.equal(a, b) for a, b in zip(filt0, filt1))
    assert set(head) == {"net.head." + n for n in HEAD_NAMES}   # only head tensors are exported / trained
    assert losses[-1] < losses[0]


def test_finetune_cli_learns_composition_classes(tmp_path):
    """Seeded random-init model (labels ~50/50 by chance), the CLI trains on the calibration draw of synth's two
    composition classes and the tuned checkpoint labels the held-out evaluation reads."""
    from chimeralm_b200 import synth
    from chimeralm_b200.engine import Engine, pack_reads
    from chimeralm_b200.weights import HEAD_PREFIX, load_checkpoint, make_state_dict

    fq = tmp_path / "train.fq"
    with fq.open("w") as f:
        i = 0
        for seqs, cls in synth.label_calibration_batches():
            for s, c in zip(seqs, cls):
                f.write(f"@read{i}|{int(c)}\n{s.tobytes().decode()}\n+\n{'I' * len(s)}\n")
                i += 1
    out = tmp_path / "tuned.ckpt"
    r = subprocess.run([sys.executable, "-m", "chimeralm_b200", "finetune", str(fq), "-o", str(out), "--epochs", "4",
                        "--lr", "1e-3", "--batch-size", "32", "--seed", "0"], cwd=ROOT, capture_output=True, text=True)
    print(r.stdout[-2000:], r.stderr[-3000:])
    assert r.returncode == 0
    tuned, base = load_checkpoint(out), make_state_dict(0)
    assert list(tuned) == list(base)
    for k in base:
        if not k.startswith(HEAD_PREFIX):
            assert torch.equal(tuned[k], base[k]), k

    def accuracy(sd):
        eng = Engine(sd, device=0, max_batch=32, max_tokens=32769)
        right = n = 0
        try:
            for seqs, cls in synth.label_eval_batches():
                T = max(len(s) for s in seqs) + 1
                bases, offs = pack_reads([s.tobytes() for s in seqs])
                ids, _ = eng.encode(bases, offs, T, add_cls=False, add_sep=True, pad_left=True, max_bases=32768)
                _, lab = eng.forward(ids, return_labels=True, check=True)
                right += int((lab.cpu().numpy() == cls).sum())
                n += len(cls)
        finally:
            eng.close()
        return right / n

    before, after = accuracy(base), accuracy(tuned)
    print(f"held-out accuracy on {2028} reads: {before:.4f} before, {after:.4f} after fine-tuning")
    assert after >= 0.95


def test_rejected_inputs(state_dict):
    from dataclasses import replace

    from chimeralm_b200 import _lib
    from chimeralm_b200.engine import Engine

    sd_mean = {k: v for k, v in state_dict.items() if ".attention." not in k}
    eng = Engine(sd_mean, device=0, cfg=replace(CFG, pooling_type="mean"), max_batch=2, max_tokens=64)
    try:
        with pytest.raises(_lib.ChimeraLMNativeError, match="attention pooling"):
            eng.head_train_begin()
    finally:
        eng.close()
    eng = Engine(state_dict, device=0, max_batch=2, max_tokens=64)
    try:
        eng.head_train_begin(lr=1e-2)
        before = eng.head_state_dict()
        ids = torch.full((2, 64), 8, dtype=torch.uint8)
        ids[1, 5] = 200
        with pytest.raises(IndexError):
            eng.head_train_step(ids.to(0), torch.tensor([0, 1]))
        after = eng.head_state_dict()
        assert all(torch.equal(before[k], after[k]) for k in before)   # a step whose forward failed changes nothing
        with pytest.raises(ValueError):
            eng.head_train_step(torch.full((2, 64), 8, dtype=torch.uint8, device=0), torch.tensor([0, 2]))
    finally:
        eng.close()


def test_classification_lit_training_step(state_dict):
    """`training_step(batch, batch_idx)` returns the batch's loss like the reference and takes an optimizer step."""
    from chimeralm_b200.model import ClassificationLit

    ids, y = _label_batch(4, 300, 600, 61)
    model = ClassificationLit(state_dict, device=0, max_batch=4, max_tokens=ids.shape[1])
    try:
        batch = {"input_ids": ids.to(0), "labels": y}
        l0 = float(model.training_step(batch, 0))
        l1 = float(model.training_step(batch, 1))
        assert np.isfinite(l0) and np.isfinite(l1) and l0 > 0
        assert model.engine.train_steps == 2
        assert model.engine.head_export("net.head.output_layer.bias").shape == (2,)
    finally:
        model.engine.close()
