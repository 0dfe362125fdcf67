"""Cost of training the last block's tail with the head, on one GPU: forward-only steps, head-only training steps and
head + tail training steps (clm_tail_train_begin), timed with CUDA events in alternating windows, at the K2 shape
(32 reads x 8 193 tokens) and at 32 reads of 1-4 kb.  Each configuration is its own engine with the same weights and
batch.  Prints one JSON line per shape with the card's name and power limit beside the numbers, and the achieved rate of
the tail's 3 538 944 FLOP per token over the difference of the two step times.

    python profiles/train_tail.py [--steps 30] [--warmup 5] [--rounds 3] [--out DIR/train_tail.json]
"""

import argparse
import json
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from chimeralm_b200 import synth  # noqa: E402
from chimeralm_b200.engine import Engine  # noqa: E402
from chimeralm_b200.weights import make_state_dict  # noqa: E402
from profiles.train_head import card, timed  # noqa: E402

TAIL_FLOP_PER_TOKEN = 3538944


def batches():
    g = torch.Generator().manual_seed(20251018)
    k2 = torch.randint(7, 11, (32, 8193), generator=g).to(torch.uint8)
    k2[:, -1] = 1
    seqs, _ = synth.label_reads(32, 7, 1000, 4000)
    short = torch.from_numpy(synth.pad_left_ids(seqs))
    y = torch.randint(0, 2, (32,), generator=g)
    return {"k2_32x8193": k2, "32_reads_1_4kb": short}, y


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sd = make_state_dict(0)
    lines = []
    shapes, y = batches()
    y = y.cuda()
    for name, ids in shapes.items():
        B, T = ids.shape
        ids = ids.cuda()
        fwd_eng = Engine(sd, device=0, max_batch=B, max_tokens=T)
        head_eng = Engine(sd, device=0, max_batch=B, max_tokens=T)
        tail_eng = Engine(sd, device=0, max_batch=B, max_tokens=T)
        head_eng.head_train_begin(lr=1e-5)
        tail_eng.head_train_begin(lr=1e-5)
        tail_eng.tail_train_begin(1e-5)
        runs = {"forward": lambda: fwd_eng.forward(ids),
                "head_step": lambda: head_eng.head_train_step(ids, y, check=False),
                "head_tail_step": lambda: tail_eng.head_train_step(ids, y, check=False)}
        for fn in runs.values():
            for _ in range(a.warmup):
                fn()
        torch.cuda.synchronize()
        ms = {k: [] for k in runs}
        for _ in range(a.rounds):   # alternate, so that clock and power drift hit all three alike
            for k, fn in runs.items():
                ms[k].append(timed(fn, a.steps))
        for e in (fwd_eng, head_eng, tail_eng):
            e.forward_status(e.last_seq)
            e.close()
        best = {k: min(v) for k, v in ms.items()}
        extra = best["head_tail_step"] - best["head_step"]
        res = {"metric": "train_tail", "gpu": card(), "shape": [B, T],
               **{f"{k}_ms": round(v, 4) for k, v in best.items()},
               "tail_extra_ms": round(extra, 4),
               "tail_tflops_over_extra": round(TAIL_FLOP_PER_TOKEN * B * T / (extra * 1e-3) / 1e12, 1) if extra > 0 else None,
               "rounds_ms": {k: [round(x, 4) for x in v] for k, v in ms.items()}}
        lines.append(json.dumps(res))
        print(lines[-1])
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
