"""Host side of training the last block's tail with the head (no GPU): the backward formulas the kernels implement
(csrc/tail_train.cuh) restated in fp64 torch against autograd, the folded-weight bookkeeping of the forward, the new
C-ABI symbol, the CLI's argument checks and the checkpoint merge."""

import re
import subprocess
import sys
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

from chimeralm_b200 import train as TR
from chimeralm_b200.config import DEFAULT_CONFIG as CFG

ROOT = Path(__file__).resolve().parents[1]
EPS = CFG.layer_norm_epsilon


def _gelu_tanh_grad(x):
    k0, k1 = 0.7978845608028654, 0.044715
    t = torch.tanh(k0 * (x + k1 * x ** 3))
    return 0.5 * (1 + t) + 0.5 * x * (1 - t * t) * k0 * (1 + 3 * k1 * x * x)


def _ln_stats(r):
    mu = r.mean(-1, keepdim=True)
    rho = 1.0 / torch.sqrt(((r - mu) ** 2).mean(-1, keepdim=True) + EPS)
    return (r - mu) * rho, rho


def test_backward_formulas_match_autograd():
    """Per row: r1 = r0 + Wo y + bo, x2 = LN2(r1), a = gelu_tanh(W1 x2 + b1), r2 = r1 + W2 a + b2, hid = ln_f(r2), then
    the head's scorer s = w2 . gelu(W0 hid + b0) + c and the pooling pooled = sum_t softmax(s)_t hid_t, with a random
    linear loss on pooled.  The hand-written backward (dhid = w dp + W0^T dz, the two LayerNorm backwards, the GELU-tanh
    derivative, the weight / bias / affine sums) equals autograd to 1e-10."""
    g = torch.Generator().manual_seed(0)
    dd = torch.float64
    T, D, DI = 37, 256, 1024

    def rnd(*s, scale=1.0):
        return torch.randn(*s, generator=g, dtype=dd) * scale

    r0, y = rnd(T, D), rnd(T, D)
    P = {"Wo": rnd(D, D, scale=D ** -0.5), "bo": rnd(D, scale=0.1), "g2": 1 + rnd(D, scale=0.1), "be2": rnd(D, scale=0.1),
         "W1": rnd(DI, D, scale=D ** -0.5), "b1": rnd(DI, scale=0.1), "W2": rnd(D, DI, scale=DI ** -0.5),
         "b2": rnd(D, scale=0.1), "gf": 1 + rnd(D, scale=0.1), "bf": rnd(D, scale=0.1)}
    W0, b0, w2 = rnd(D, D, scale=D ** -0.5), rnd(D, scale=0.1), rnd(D, scale=0.3)
    dp = rnd(D)
    prm = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    r1 = r0 + F.linear(y, prm["Wo"], prm["bo"])
    x2 = F.layer_norm(r1, (D,), prm["g2"], prm["be2"], EPS)
    h = F.linear(x2, prm["W1"], prm["b1"])
    r2 = r1 + F.linear(F.gelu(h, approximate="tanh"), prm["W2"], prm["b2"])
    hid = F.layer_norm(r2, (D,), prm["gf"], prm["bf"], EPS)
    s = F.gelu(F.linear(hid, W0, b0)) @ w2
    w = torch.softmax(s, 0)
    loss = (w[:, None] * hid).sum(0) @ dp
    loss.backward()

    with torch.no_grad():
        # forward restated, with the folded weights the kernels read
        r1 = r0 + y @ P["Wo"].T + P["bo"]
        n1, rho1 = _ln_stats(r1)
        W1f, b1f = P["W1"] * P["g2"] / 2, (P["b1"] + P["W1"] @ P["be2"]) / 2   # W1' = W1 diag(g2) / 2, b1' halved too
        hh = n1 @ W1f.T + b1f
        x2 = P["g2"] * n1 + P["be2"]
        h = x2 @ P["W1"].T + P["b1"]
        assert torch.allclose(2 * hh, h, rtol=0, atol=1e-10)
        a = F.gelu(h, approximate="tanh")
        r2 = r1 + a @ P["W2"].T + P["b2"]
        n2, rho2 = _ln_stats(r2)
        W0f, b0f = W0 * P["gf"], b0 + W0 @ P["bf"]   # ln_f folded into the scorer
        z = n2 @ W0f.T + b0f
        assert torch.allclose(z, (P["gf"] * n2 + P["bf"]) @ W0.T + b0, rtol=0, atol=1e-10)
        hid = P["gf"] * n2 + P["bf"]
        # backward as the kernels form it
        s = F.gelu(z) @ w2
        wt = torch.softmax(s, 0)
        pooled = (wt[:, None] * hid).sum(0)
        ds = wt * ((hid - pooled) @ dp)
        phi = torch.exp(-0.5 * z * z) / (2 * torch.pi) ** 0.5
        dz = ds[:, None] * w2 * (0.5 * (1 + torch.erf(z / 2 ** 0.5)) + z * phi)
        dhid = wt[:, None] * dp + dz @ W0
        dn2 = P["gf"] * dhid
        dr2 = rho2 * (dn2 - dn2.mean(-1, keepdim=True) - n2 * (dn2 * n2).mean(-1, keepdim=True))
        dh = (dr2 @ P["W2"]) * _gelu_tanh_grad(h)
        dx2 = dh @ P["W1"]
        dn1 = P["g2"] * dx2
        dr1 = dr2 + rho1 * (dn1 - dn1.mean(-1, keepdim=True) - n1 * (dn1 * n1).mean(-1, keepdim=True))
        mine = {"gf": (dhid * n2).sum(0), "bf": dhid.sum(0), "W2": dr2.T @ a, "b2": dr2.sum(0), "W1": dh.T @ x2,
                "b1": dh.sum(0), "g2": (dx2 * n1).sum(0), "be2": dx2.sum(0), "Wo": dr1.T @ y, "bo": dr1.sum(0)}
    for k, v in mine.items():
        ref = prm[k].grad
        assert float((v - ref).abs().max()) <= 1e-10 * max(1.0, float(ref.abs().max())), k


def test_tail_keys_and_parameter_count():
    from chimeralm_b200.engine import tail_keys
    from chimeralm_b200.weights import make_state_dict

    keys = tail_keys(CFG.n_layer)
    sd = make_state_dict(0)
    assert len(keys) == 10 and all(k in sd for k in keys)
    assert keys[0] == "net.backbone.backbone.layers.3.mixer.out_proj.weight"
    assert sum(sd[k].numel() for k in keys) == 592384


def test_symbol_and_ctypes_signature():
    import ctypes as C

    from chimeralm_b200 import _lib

    res, args = _lib._SIGNATURES["clm_tail_train_begin"]
    assert res is C.c_int and args == [C.c_void_p, C.c_float]
    hdr = (ROOT / "include" / "chimeralm_b200.h").read_text()
    assert re.search(r"int clm_tail_train_begin\(clm_ctx\* ctx, float lr\);", hdr)


def test_cli_rejects_tail_lr_without_train_tail(tmp_path):
    fq = tmp_path / "t.fq"
    fq.write_text("@a|0\nACGT\n+\nIIII\n")
    r = subprocess.run([sys.executable, "-m", "chimeralm_b200", "finetune", str(fq), "-o", str(tmp_path / "o.ckpt"),
                        "--tail-lr", "1e-4"], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 1 and "--tail-lr needs --train-tail" in r.stdout + r.stderr
    r = subprocess.run([sys.executable, "-m", "chimeralm_b200", "finetune", "--help"], cwd=ROOT, capture_output=True,
                       text=True)
    assert r.returncode == 0 and "--train-tail" in r.stdout and "--tail-lr" in r.stdout
    with pytest.raises(ValueError, match="--tail-lr needs --train-tail"):
        TR.finetune(fq, None, tmp_path / "o.ckpt", tail_lr=1e-4)
    with pytest.raises(ValueError, match="tail_lr needs train_tail"):
        TR.fit(None, [], [], tail_lr=1e-4)


class _FakeEngine:
    def __init__(self, head, tail):
        self.head, self.tail = head, tail

    def head_state_dict(self):
        return self.head

    def tail_state_dict(self):
        return self.tail


def test_checkpoint_merge_replaces_exactly_the_trained_keys():
    from chimeralm_b200.engine import tail_keys
    from chimeralm_b200.weights import HEAD_PREFIX, make_state_dict

    sd = make_state_dict(3)
    head = {k: v + 1.0 for k, v in sd.items() if k.startswith(HEAD_PREFIX)}
    tail = {k: sd[k] + 2.0 for k in tail_keys(CFG.n_layer)}
    eng = _FakeEngine(head, tail)
    for train_tail, n in ((True, 24), (False, 14)):
        out = TR.tuned_state_dict(sd, eng, train_tail=train_tail)
        assert list(out) == list(sd)
        changed = {k for k in sd if not torch.equal(out[k], sd[k])}
        assert len(changed) == n and changed == set(head) | (set(tail) if train_tail else set())
