"""Cost of evaluation against the forward on one GPU: clm_eval_step (forward + per-read loss and probability) and
clm_forward on the same batch, timed with CUDA events in alternating windows after a warm-up, at the K2 shape (32 reads x
8 193 tokens) and at a batch of 32 reads of 1-4 kb (synth.label_reads, left-padded to the longest).  Prints one JSON
line with the card's name and power limit beside the numbers.

    python profiles/eval_head.py [--steps 50] [--warmup 10] [--rounds 3] [--out DIR/eval_head.json]
"""

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from chimeralm_b200 import synth  # noqa: E402
from chimeralm_b200.engine import Engine  # noqa: E402
from chimeralm_b200.weights import make_state_dict  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def timed(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def shapes():
    g = torch.Generator().manual_seed(20251018)
    k2 = torch.randint(7, 11, (32, 8193), generator=g).to(torch.uint8)
    k2[:, -1] = 1
    seqs, _ = synth.label_reads(32, 4242, 1000, 4000)
    short = torch.from_numpy(synth.pad_left_ids(seqs))
    y = torch.randint(0, 2, (32,), generator=g)
    return {"k2_32x8193": (k2, y), "reads_1_4kb_32": (short, y)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    eng = Engine(make_state_dict(0), device=0, max_batch=32, max_tokens=8193)
    res = {"metric": "eval_step_vs_forward", "gpu": card(), "steps": a.steps, "rounds": a.rounds}
    for name, (ids, y) in shapes().items():
        ids, y = ids.cuda(), y.cuda()
        fwd = lambda: eng.forward(ids)                       # noqa: E731
        ev = lambda: eng.eval_step(ids, y, check=False)      # noqa: E731
        for _ in range(a.warmup):
            fwd()
            ev()
        torch.cuda.synchronize()
        eng.forward_status(eng.last_seq)
        f_ms, e_ms = [], []
        for _ in range(a.rounds):   # alternate the two, so that clock and power drift hit both alike
            f_ms.append(timed(fwd, a.steps))
            e_ms.append(timed(ev, a.steps))
        eng.forward_status(eng.last_seq)
        # device time of the loss / probability kernel alone: per-launch CUDA events, in a run of their own
        eng.profile(True)
        eng.profile_reset()
        for _ in range(10):
            ev()
        prof = eng.profile_read()
        eng.profile(False)
        fm, em = min(f_ms), min(e_ms)
        res[name] = {"shape": list(ids.shape), "forward_ms": round(fm, 4), "eval_step_ms": round(em, 4),
                     "eval_over_forward": round(em / fm, 4), "eval_reads_per_s": round(ids.shape[0] / em * 1e3, 1),
                     "rounds_forward_ms": [round(x, 4) for x in f_ms], "rounds_eval_ms": [round(x, 4) for x in e_ms],
                     "eval_rows_kernel_ms": round(prof["eval"][0] / prof["eval"][1], 5)}
    eng.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
