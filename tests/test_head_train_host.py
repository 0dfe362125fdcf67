"""Host side of head fine-tuning (no GPU): labels from read ids, the dropout-mask mirror, the AdamW arithmetic and the
tuned checkpoint."""

import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from chimeralm_b200 import train as TR

ROOT = Path(__file__).resolve().parents[1]


def test_parse_target():
    assert TR.parse_target("3f2a-uuid|0") == 0
    assert TR.parse_target("3f2a-uuid|1") == 1
    assert TR.parse_target("m64011/1/ccs;x|y|1") == 1     # the label is the last field
    assert TR.parse_target("read") is None                 # no suffix: no label
    assert TR.parse_target("read|") is None
    assert TR.parse_target("read|chimeric") is None


def test_unlabelled_reads_are_rejected_for_training(tmp_path):
    fq = tmp_path / "t.fq"
    fq.write_text("@a|0\nACGT\n+\nIIII\n@b\nACGA\n+\nIIII\n")
    with pytest.raises(ValueError, match="no 0/1 label"):
        TR.read_labelled(fq)
    fq.write_text("@a|0 desc\nacgt\n+\nIIII\n@b|1\nACGA\n+\nIIII\n")
    names, seqs, labels = TR.read_labelled(fq)
    assert names == ["a|0", "b|1"] and labels.tolist() == [0, 1] and seqs[0].tobytes() == b"ACGT"


def test_dropout_mask_rate_and_independence():
    p, B, H = 0.1, 64, 512
    m = TR.dropout_masks(seed=7, step=0, B=B, p=p, hidden=H)
    assert m.shape == (3, B, H) and m.dtype == bool
    n = B * H
    for site in range(3):   # dropped fraction within 5 standard deviations of the binomial
        drop = 1.0 - m[site].mean()
        assert abs(drop - p) < 5 * np.sqrt(p * (1 - p) / n), (site, drop)
    assert not np.array_equal(m[0], m[1]) and not np.array_equal(m[1], m[2])
    m1 = TR.dropout_masks(seed=7, step=1, B=B, p=p, hidden=H)
    assert not np.array_equal(m, m1)
    assert np.array_equal(m, TR.dropout_masks(seed=7, step=0, B=B, p=p, hidden=H))
    assert not np.array_equal(m, TR.dropout_masks(seed=8, step=0, B=B, p=p, hidden=H))
    assert TR.dropout_masks(seed=7, step=0, B=4, p=0.0).all()
    # different reads and units see different bits (no row or column repeats)
    assert len({r.tobytes() for r in m[0]}) == B


def test_dropout_mirror_matches_the_device_hash(tmp_path):
    """The numpy mirror against the very function the kernels call (dropout_keep of csrc/head_train.cuh, compiled for
    the host)."""
    src = tmp_path / "h.cu"
    src.write_text('#include <cstdio>\n#include "head_train.cuh"\n'
                   "int main() { for (unsigned st = 0; st < 3; ++st) for (unsigned s = 0; s < 3; ++s)"
                   " for (unsigned b = 0; b < 5; ++b) for (unsigned u = 0; u < 512; ++u)"
                   " putchar(clm::dropout_keep(12345u, st, s, b, u, 1677722u) ? '1' : '0'); return 0; }\n")
    exe = tmp_path / "h"
    subprocess.run(["/usr/local/cuda/bin/nvcc", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-I",
                    str(ROOT / "chimeralm_b200" / "csrc"), "-o", str(exe), str(src)], check=True)
    got = np.frombuffer(subprocess.run([str(exe)], check=True, capture_output=True).stdout, np.uint8) == ord("1")
    want = np.stack([TR.dropout_masks(12345, st, 5, 0.1) for st in range(3)]).reshape(-1)
    assert TR.dropout_threshold(0.1) == 1677722
    assert np.array_equal(got, want)


def test_adamw_arithmetic_matches_torch():
    rng = np.random.default_rng(0)
    shapes = [(64, 32), (512,), (1,)]
    ps = [torch.from_numpy(rng.standard_normal(s).astype(np.float32)) for s in shapes]
    params = [torch.nn.Parameter(p.clone()) for p in ps]
    hp = dict(lr=3e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)
    opt = torch.optim.AdamW(params, foreach=False, **hp)
    mine = [(p.numpy().copy(), np.zeros(p.shape, np.float32), np.zeros(p.shape, np.float32)) for p in ps]
    for t in range(1, 6):
        grads = [rng.standard_normal(s).astype(np.float32) * (10.0 ** -t) for s in shapes]
        for prm, g in zip(params, grads):
            prm.grad = torch.from_numpy(g.copy())
        opt.step()
        mine = [TR.adamw_update(p, g, m, v, t, **hp) for (p, m, v), g in zip(mine, grads)]
        for prm, (p, _, _) in zip(params, mine):
            ref = prm.detach().numpy()
            assert np.linalg.norm(p - ref) <= 1e-6 * np.linalg.norm(ref), t


class _FakeEngine:
    def __init__(self, head):
        self.head = head

    def head_state_dict(self):
        return self.head


def test_tuned_checkpoint_round_trip(tmp_path):
    from chimeralm_b200.weights import HEAD_PREFIX, load_checkpoint, make_state_dict, save_lightning_ckpt

    sd = make_state_dict(3)
    head = {k: v + 1.0 for k, v in sd.items() if k.startswith(HEAD_PREFIX)}
    out = TR.tuned_state_dict(sd, _FakeEngine(head))
    assert list(out) == list(sd)
    save_lightning_ckpt(out, tmp_path / "tuned.ckpt")
    back = load_checkpoint(tmp_path / "tuned.ckpt")
    assert list(back) == list(sd)
    for k, v in sd.items():
        if k.startswith(HEAD_PREFIX):
            assert torch.equal(back[k], v + 1.0), k
        else:
            assert torch.equal(back[k], v), k   # backbone bit-identical
