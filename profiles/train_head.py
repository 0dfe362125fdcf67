"""Head fine-tuning throughput at the K2 shape (32 reads x 8 193 tokens) on one GPU: training steps per second
(clm_head_train_step: forward + classifier with dropout + loss + head backward + AdamW + refresh) against forward-only
steps, timed with CUDA events in alternating windows, plus the device time of the backward kernels alone.  Prints one JSON
line with the card's name and power limit beside the numbers.

    python profiles/train_head.py [--steps 50] [--warmup 10] [--out DIR/train_head.json]
"""

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    B, T = 32, 8193
    eng = Engine(make_state_dict(0), device=0, max_batch=B, max_tokens=T)
    g = torch.Generator().manual_seed(20251018)
    ids = torch.randint(7, 11, (B, T), generator=g).to(torch.uint8)
    ids[:, -1] = 1
    ids = ids.cuda()
    y = torch.randint(0, 2, (B,), generator=g).cuda()
    eng.head_train_begin(lr=1e-4)
    fwd = lambda: eng.forward(ids)                             # noqa: E731
    step = lambda: eng.head_train_step(ids, y, check=False)    # noqa: E731
    for _ in range(a.warmup):
        fwd()
        step()
    torch.cuda.synchronize()
    f_ms, s_ms = [], []
    for _ in range(a.rounds):   # alternate the two, so that clock and power drift hit both alike
        f_ms.append(timed(fwd, a.steps))
        s_ms.append(timed(step, a.steps))
    eng.forward_status(eng.last_seq)
    # device time per kernel class of a training step (head_train = everything after the forward), per-launch CUDA
    # events in a run of their own: the events slow the host
    eng.profile(True)
    eng.profile_reset()
    for _ in range(5):
        step()
    prof = eng.profile_read()
    eng.profile(False)
    eng.close()
    fm, sm = min(f_ms), min(s_ms)
    res = {"metric": "head_train_k2", "gpu": card(), "shape": [B, T],
           "forward_ms": round(fm, 4), "train_step_ms": round(sm, 4), "train_over_forward": round(sm / fm, 3),
           "forward_reads_per_s": round(B / fm * 1e3, 1), "train_reads_per_s": round(B / sm * 1e3, 1),
           "train_steps_per_s": round(1e3 / sm, 2), "rounds_forward_ms": [round(x, 4) for x in f_ms],
           "rounds_train_ms": [round(x, 4) for x in s_ms],
           "train_step_kernel_classes_ms_per_step": {k: round(v[0] / 5, 4) for k, v in prof.items()}}
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
