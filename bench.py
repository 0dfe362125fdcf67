#!/usr/bin/env python
"""Headline benchmark: `chimeralm predict` throughput (reads/s) on synthetic long reads.

Contract (see the task brief): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line.

  value / e2e     K2 (BASELINE.json configs[1]): 8 192-base reads, batch 32 per GPU, T = 8 193.  A step = one batch
                  through the predict hot path (tokenise -> forward -> labels).  `value` has the read bytes resident
                  in HBM; `e2e` goes through the C-ABI host entry point (`clm_predict_host`) with pinned HOST buffers,
                  H2D and D2H inside the timed region.  Timed with CUDA events, max over ranks, the final NCCL
                  all_gather of labels inside the region (warmed once before it, and also timed on its own).
  roofline        dominant kernel class, from a SECOND, profiled pass over the same steps (`clm_profile_*`: CUDA
                  events on the launching stream around every launch) so the profiling never sits inside `value`.
  k3              configs[2..3]: log-normal 1-32 kb reads (seed 20251019), length-bucketed into batches of <= 256
                  reads / <= 262 176 padded tokens; at N > 1 (= K4) the batches are dealt to the ranks by greedy LPT on
                  the batch cost model and the (index, label) pairs are gathered at the end.  Strong scaling: the
                  sample is fixed, `value` = sample reads / slowest rank's time.  Unpadded bases/s and padding waste
                  are reported, because throughput counts real bases.
  k5              configs[4]: reads of exactly 32 768 bases (T = 32 769), batch 64 per GPU, weak scaling.
  label_agreement argmax labels vs the CPU oracle's golden logits on the 2 028-read label set (tests/golden/
                  label_agreement.npz; probe head, see oracle/make_label_golden.py), rank 0.
  cpu_baseline    the reference-equivalent CPU predict path (oracle port) on a bounded sample, rank 0.

`--impl reference` times that CPU path alone on the same workload definition.

`--dump-outputs DIR` writes what the `value` pass returned in its last timed step on rank 0 - logits [B, 2] and labels
[B] - as DIR/logits.npy and DIR/labels.npy (float32).  Inputs and weights are seeded, so two builds run with the same
arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import datetime
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

from chimeralm_b200 import synth  # noqa: E402

READ_LEN = 8192          # K2: fixed 8 kb reads
BATCH = 32               # K2: batch 32
N_DISTINCT = 8           # distinct synthetic batches rotated through the timed region
F_TOK = 6_423_040        # dense FLOP/token of the reference's graph (SURVEY.md 8(d))
# ... of which block 0's in_proj (2 x 256 x 768) is NOT executed as a GEMM here: its input is one of 16 embedding rows, so the
# product is a table lookup (csrc/embed_in.cuh).  The dense_tensor_* figures count executed tensor work only.
F_TOK_EXEC = F_TOK - 2 * 256 * 768
CONV_BYTES_TOK_LAYER = 1536  # long-conv algorithmic bytes/token/layer (vx in, x0 in, y*x0 out; 2 B each x 256 channels)
K3_TOKEN_CAP = BATCH * (READ_LEN + 1)   # padded tokens per bucketed batch: the K2 step's size
K3_MAX_READS = 256
ENC = dict(add_cls=False, add_sep=True, pad_left=True, max_bases=32768)


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"],
                "tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1590.0, "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """`nvidia-smi -lms 20` on one GPU, started early (nvidia-smi needs up to a second to come up on an 8-GPU box);
    rows are time-stamped and reported per named window [mark_start, mark_end]."""
    QUERY = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.windows = {}
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def mark_start(self, name="k2"):
        self.windows[name] = [datetime.datetime.now(), None]

    def mark_end(self, name="k2"):
        self.windows[name][1] = datetime.datetime.now()

    def stop(self):
        empty = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return {k: dict(empty) for k in self.windows}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [r.split(", ") for r in Path(self.f.name).read_text().strip().splitlines() if r.count(",") >= 9]
        os.unlink(self.f.name)

        def when(r):
            try:
                return datetime.datetime.strptime(r[0].strip(), "%Y/%m/%d %H:%M:%S.%f")
            except ValueError:
                return None

        out = {}
        for name, (t0, t1) in self.windows.items():
            o = dict(empty)
            inside = [r for r in rows if t0 and t1 and when(r) and t0 <= when(r) <= t1]
            if inside:
                o["window"] = "timed region"
            else:  # region shorter than the sampling period: the samples taken under load closest to it
                before_end = [r for r in rows if t1 and when(r) and when(r) <= t1]
                inside = before_end[-3:] or rows[-3:]
                o["window"] = "last samples up to the end of the timed region (region shorter than the 20 ms sampling period)"
            if inside:
                sm = sorted(float(r[2]) for r in inside)
                o["sm_mhz"] = sm[len(sm) // 2]
                o["sm_mhz_min"] = sm[0]
                o["sm_max_mhz"] = float(inside[0][3])
                o["power_w_max"] = max(float(r[4]) for r in inside)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                o["reasons"] = [n for i, n in enumerate(names) if any(r[6 + i].strip().lower().startswith("active") for r in inside)]
                o["samples"] = len(inside)
            out[name] = o
        return out


def workload_config(L, T, B, world):
    tokens_per_step = B * T
    return {"workload": f"K2: synthetic {L} b reads, T={T} tokens (ids+[SEP]), batch {B} per GPU, random-init ChimeraLM",
            "read_len": L, "batch_per_gpu": B, "parallelism": f"dp{world} (reads sharded, final all_gather of labels)",
            "l2": f"per-step activation working set ~{tokens_per_step * 256 * 12 / 1e6:.0f} MB >> 126 MB L2; {N_DISTINCT} distinct input batches rotate"}


def cpu_reference_path(sd, cfg, seqs_ascii: np.ndarray, batch: int = 12):
    """Reference-equivalent CPU predict on `seqs_ascii` [n, L] (chimeralm/__main__.py:248-319
    pipeline restated): per-read Python tokeniser -> collate (left pad) -> fp32 forward -> argmax."""
    from oracle import hyena_oracle, tokenizer_oracle

    n = seqs_ascii.shape[0]
    t0 = time.perf_counter()
    rows = [tokenizer_oracle.encode(bytes(r).decode(), max_length=32769, add_cls=False) for r in seqs_ascii]
    t_tok = time.perf_counter() - t0
    labels = []
    t1 = time.perf_counter()
    for i in range(0, n, batch):
        ids = torch.tensor(tokenizer_oracle.collate(rows[i:i + batch], padding_side="left"), dtype=torch.int64)
        labels += hyena_oracle.predict_labels(sd, ids, cfg).tolist()
    t_fwd = time.perf_counter() - t1
    return n / (t_tok + t_fwd), t_tok, t_fwd, labels


def run_reference(args, sd, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    # one step = one batch of the SAME workload (batch 32 x 8 192 b) through the CPU path, ~4 s on 16 cores; with many
    # steps requested the per-step sample shrinks to the reference CLI's default batch of 12 so the run stays bounded
    n_per_step = args.batch if args.steps + args.warmup <= 30 else 12
    reads = synth.uniform_reads(n_per_step * max(1, min(args.steps + args.warmup, 4)), args.read_len, synth.K2_SEED)
    for w in range(args.warmup):
        cpu_reference_path(sd, cfg, reads[:n_per_step], batch=n_per_step)
    t0 = time.perf_counter()
    for s in range(args.steps):
        off = (s % (reads.shape[0] // n_per_step)) * n_per_step
        cpu_reference_path(sd, cfg, reads[off:off + n_per_step], batch=n_per_step)
    dt = time.perf_counter() - t0
    val = n_per_step * args.steps / dt
    line = {
        "impl": "reference", "metric": "predict_reads_per_s", "value": val, "unit": "reads/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.read_len, args.read_len + 1, args.batch, max(1, args.gpus)),
        "bases_per_s": val * args.read_len,
        "cpu_baseline": {"value": val, "unit": "reads/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"each step = one batch of {n_per_step} reads x {args.read_len} b of the same synthetic workload through the "
                                   f"CPU predict path (python tokeniser, collate, fp32 eager forward, argmax); {args.steps} steps; rank 0 only"},
        "e2e": {"value": val, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
class Dist:
    """torch.distributed plumbing (NCCL) with the N = 1 case folded in."""

    def __init__(self, local_rank):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.dev = torch.device("cuda", local_rank)
        self.pg = None
        if self.world > 1:
            import torch.distributed as dist

            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
            self.pg = dist

    def barrier(self):
        torch.cuda.synchronize()
        if self.pg is not None:
            self.pg.barrier()
        torch.cuda.synchronize()

    def all_gather(self, t):
        if self.pg is None:
            return [t]
        out = [torch.empty_like(t) for _ in range(self.world)]
        self.pg.all_gather(out, t)
        return out

    def gather_floats(self, vals):
        """list of per-rank float lists (every rank contributes len(vals) numbers)"""
        t = torch.tensor(vals, dtype=torch.float64, device=self.dev)
        return [x.tolist() for x in self.all_gather(t)]

    def close(self):
        if self.pg is not None:
            self.pg.destroy_process_group()
            self.pg = None


def e2e_pipelined(eng, items, max_reads):
    """Batches from pinned HOST memory through the C-ABI's submit / wait pair with up to 3 in flight: H2D, encode, forward
    and D2H of every batch are inside the caller's timed region; returns when the last batch's labels are on the host."""
    from collections import deque

    lo = [torch.empty(max_reads, 2, dtype=torch.float32).pin_memory() for _ in range(3)]
    la = [torch.empty(max_reads, dtype=torch.uint8).pin_memory() for _ in range(3)]
    pending = deque()
    for i, (hb, ho, T, B) in enumerate(items):
        pending.append(eng.predict_host_submit(hb, ho, T, logits_out=lo[i % 3][:B], labels_out=la[i % 3][:B], **ENC))
        if len(pending) == 3:
            eng.predict_host_wait(pending.popleft())
    while pending:
        eng.predict_host_wait(pending.popleft())
    return lo, la


def run_k2(args, eng, D, sampler):
    B, L = args.batch, args.read_len
    T = L + 1
    reads = synth.uniform_reads(N_DISTINCT * B, L, synth.K2_SEED + D.rank)   # each rank its own shard (weak scaling)
    offsets_h = torch.arange(0, (B + 1) * L, L, dtype=torch.int64)
    dev_batches = [torch.from_numpy(reads[i * B:(i + 1) * B].reshape(-1).copy()).to(D.dev) for i in range(N_DISTINCT)]
    host_batches = [torch.from_numpy(reads[i * B:(i + 1) * B].reshape(-1).copy()).pin_memory() for i in range(N_DISTINCT)]
    offsets_d, offsets_p = offsets_h.to(D.dev), offsets_h.pin_memory()

    def step_resident(i):
        ids, _ = eng.encode(dev_batches[i % N_DISTINCT], offsets_d, T, **ENC)
        return eng.forward(ids, return_labels=True)

    def timed_pass():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        labels = []
        ev[0].record()
        for i in range(args.steps):
            last = step_resident(i)
            labels.append(last[1])
        mine = torch.cat(labels)
        ev[1].record()
        D.all_gather(mine)   # the path's only exchange: final gather of predictions
        ev[2].record()
        return ev, last

    def settle():
        # The board reaches its power cap within a few tenths of a second of this load and then drops from 1 965 MHz to
        # 1 700-1 850 MHz (profiles/r2_e2e_gap.txt).  Every timed pass therefore starts from the same state: one second of
        # idle, then the W warm-up steps - otherwise whichever pass happens to run first gets the higher clock.
        torch.cuda.synchronize()
        time.sleep(1.0)

    # ---- `e2e`: through the C-ABI host entry point, H2D + D2H inside
    settle()
    for i in range(args.warmup):
        step_resident(i)
    e2e_pipelined(eng, [(host_batches[i % N_DISTINCT], offsets_p, T, B) for i in range(args.warmup)], B)
    D.barrier()
    if sampler:
        sampler.mark_start("k2_e2e")
    t0 = time.perf_counter()
    e2e_pipelined(eng, [(host_batches[i % N_DISTINCT], offsets_p, T, B) for i in range(args.steps)], B)
    e2e_s = time.perf_counter() - t0
    if sampler:
        sampler.mark_end("k2_e2e")
    # and the plain synchronous call, one batch at a time (what a caller without a pipeline gets)
    lo = torch.empty(B, 2, dtype=torch.float32).pin_memory()
    settle()
    for i in range(args.warmup):
        eng.predict_host(host_batches[i % N_DISTINCT], offsets_p, T, logits_out=lo, **ENC)
    D.barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        eng.predict_host(host_batches[i % N_DISTINCT], offsets_p, T, logits_out=lo, **ENC)
    e2e_sync_s = time.perf_counter() - t0
    # ---- `value`: device-resident, un-profiled
    settle()
    for i in range(args.warmup):
        step_resident(i)
    D.all_gather(torch.zeros(args.steps * B, dtype=torch.uint8, device=D.dev))   # NCCL's first collective of this shape is not a step
    D.barrier()
    if sampler:
        sampler.mark_start("k2")
    launches0 = eng.launch_count
    ev, (logits, labels) = timed_pass()
    D.barrier()
    if sampler:
        sampler.mark_end("k2")
    ms, gather_ms = ev[0].elapsed_time(ev[2]), ev[1].elapsed_time(ev[2])
    launches = eng.launch_count - launches0
    assert eng.forward_status() is None

    # ---- second pass with per-launch CUDA events: kernel times for the roofline (not part of `value`)
    settle()
    for i in range(args.warmup):
        step_resident(i)
    D.barrier()
    eng.profile_reset()
    eng.profile(True)
    evp, _ = timed_pass()
    D.barrier()
    prof = eng.profile_read()
    eng.profile(False)
    ms_prof = evp[0].elapsed_time(evp[2])
    kernel_sum = sum(v[0] for v in prof.values())

    # ---- the same two measurements in the STEADY state: ~1.5 s of the same load first, so the board is at its power cap
    # (1 700-1 850 MHz) when the K timed steps run.  `value` / `e2e` above start one second after idle and see boost clocks;
    # an 8-GPU box runs every rank at the capped clock from the start, so the scaling of the steady-state figures is the
    # like-for-like one.
    def preheat(seconds):
        t_end = time.perf_counter() + seconds
        i = 0
        while time.perf_counter() < t_end:
            for _ in range(8):
                step_resident(i)
                i += 1
            torch.cuda.synchronize()

    preheat(args.preheat)
    D.barrier()
    if sampler:
        sampler.mark_start("k2_steady")
    evs, _ = timed_pass()
    D.barrier()
    if sampler:
        sampler.mark_end("k2_steady")
    ms_steady = evs[0].elapsed_time(evs[2])
    preheat(args.preheat / 3)
    D.barrier()
    t0 = time.perf_counter()
    e2e_pipelined(eng, [(host_batches[i % N_DISTINCT], offsets_p, T, B) for i in range(args.steps)], B)
    e2e_steady_s = time.perf_counter() - t0
    per_rank = D.gather_floats([ms, gather_ms, ms_prof, kernel_sum, e2e_s * 1e3, e2e_sync_s * 1e3, ms_steady, e2e_steady_s * 1e3])
    return {"B": B, "L": L, "T": T, "prof": prof, "launches": launches, "per_rank": per_rank,
            "outputs": {"logits": logits, "labels": labels}}


def run_k5(args, eng, D, sampler):
    """K5: 32 768-base reads (T = 32 769), batch 64 per GPU, >= 16 batches per GPU; weak scaling."""
    B, L = args.k5_batch, 32768
    T = L + 1
    eng.reserve(B, T)
    reads = synth.uniform_reads(2 * B, L, synth.K5_SEED + D.rank)
    offsets_d = torch.arange(0, (B + 1) * L, L, dtype=torch.int64, device=D.dev)
    dev_batches = [torch.from_numpy(reads[i * B:(i + 1) * B].reshape(-1).copy()).to(D.dev) for i in range(2)]
    host_batches = [torch.from_numpy(reads[i * B:(i + 1) * B].reshape(-1).copy()).pin_memory() for i in range(2)]
    offsets_p = torch.arange(0, (B + 1) * L, L, dtype=torch.int64).pin_memory()

    def step(i):
        ids, _ = eng.encode(dev_batches[i % 2], offsets_d, T, **ENC)
        return eng.forward(ids, return_labels=True)[1]

    for i in range(2):
        step(i)
    D.all_gather(torch.zeros(args.k5_steps * B, dtype=torch.uint8, device=D.dev))
    D.barrier()
    if sampler:
        sampler.mark_start("k5")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    labels = [step(i) for i in range(args.k5_steps)]
    D.all_gather(torch.cat(labels))
    ev1.record()
    D.barrier()
    if sampler:
        sampler.mark_end("k5")
    ms = ev0.elapsed_time(ev1)
    assert eng.forward_status() is None
    eng.profile_reset()
    eng.profile(True)
    for i in range(2):
        step(i)
    torch.cuda.synchronize()
    prof = eng.profile_read()
    eng.profile(False)
    e2e_pipelined(eng, [(host_batches[0], offsets_p, T, B)], B)
    D.barrier()
    t0 = time.perf_counter()
    n_e2e = max(3, args.k5_steps // 2)
    e2e_pipelined(eng, [(host_batches[i % 2], offsets_p, T, B) for i in range(n_e2e)], B)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / n_e2e
    per_rank = D.gather_floats([ms, e2e_ms])
    ms_max = max(r[0] for r in per_rank)
    reads_s = D.world * B * args.k5_steps / (ms_max / 1e3)
    return {"workload": f"K5: {L} b reads, T={T}, batch {B} per GPU, {args.k5_steps} batches per GPU, weak scaling",
            "reads_per_s": reads_s, "bases_per_s": reads_s * L, "tokens_per_s": reads_s * T, "ms_per_step": ms_max / args.k5_steps,
            "ms_per_rank": [r[0] for r in per_rank],
            "e2e_reads_per_s": D.world * B / (max(r[1] for r in per_rank) / 1e3),
            "dense_tensor_frac_of_burst_peak": F_TOK_EXEC * reads_s / D.world * T / 1e12 / peaks()["tflops_burst"],
            "longconv_kernel": eng.longconv_variant(T),
            "kernel_ms_per_step": {k: v[0] / 2 for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}}


def run_k3(args, eng, D, sampler):
    """K3 (N = 1) / K4 (N > 1): log-normal 1-32 kb reads, length-bucketed, token-balanced LPT dealing, final gather."""
    n = args.k3_reads
    flat, offsets = synth.k3_reads(n)
    lens = np.diff(offsets)
    batches = synth.bucket_batches(lens, K3_MAX_READS, n_special=1, max_tokens_per_batch=K3_TOKEN_CAP)
    shapes = [(len(b), int(lens[b].max()) + 1) for b in batches]
    costs = [synth.batch_cost(B, T) for B, T in shapes]
    ranks, loads = synth.deal_lpt(costs, D.world)
    mine = ranks[D.rank]
    eng.reserve(K3_MAX_READS, 32769, K3_TOKEN_CAP)
    staged = []
    for bi in mine:   # assemble this rank's batches: contiguous bases + offsets, pinned on the host and resident on the device
        idx = batches[bi]
        offs = np.zeros(len(idx) + 1, np.int64)
        np.cumsum(lens[idx], out=offs[1:])
        bases = np.concatenate([flat[offsets[i]:offsets[i + 1]] for i in idx])
        hb, ho = torch.from_numpy(bases).pin_memory(), torch.from_numpy(offs).pin_memory()
        staged.append((bi, hb, ho, hb.to(D.dev), ho.to(D.dev), shapes[bi]))
    my_reads = sum(s[5][0] for s in staged)
    my_tokens = sum(int(lens[batches[s[0]]].sum()) + s[5][0] for s in staged)
    my_padded = sum(s[5][0] * s[5][1] for s in staged)
    n_max = max(sum(shapes[b][0] for b in r) for r in ranks)

    def resident(s):
        ids, _ = eng.encode(s[3], s[4], s[5][1], **ENC)
        return eng.forward(ids, return_labels=True)[1]

    for s in (staged[:: max(1, len(staged) // 6)] + staged[-1:]):   # warm every kernel variant the sample uses
        resident(s)
    D.all_gather(torch.zeros(n_max, 2, dtype=torch.int32, device=D.dev))
    D.barrier()
    if sampler:
        sampler.mark_start("k3")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    labels = [resident(s) for s in staged]
    pairs = torch.zeros(n_max, 2, dtype=torch.int32, device=D.dev)   # (read index, label), padded to the largest rank
    if staged:
        idx_dev = torch.from_numpy(np.concatenate([batches[s[0]] for s in staged]).astype(np.int32)).to(D.dev, non_blocking=True)
        pairs[:my_reads, 0] = idx_dev
        pairs[:my_reads, 1] = torch.cat(labels).to(torch.int32)
    pairs[my_reads:, 0] = -1
    ev[1].record()
    gathered = D.all_gather(pairs)
    ev[2].record()
    D.barrier()
    if sampler:
        sampler.mark_end("k3")
    ms, gather_ms = ev[0].elapsed_time(ev[2]), ev[1].elapsed_time(ev[2])
    assert eng.forward_status() is None
    got = torch.cat(gathered)[:, 0]
    assert sorted(got[got >= 0].tolist()) == list(range(n)), "every read must come back exactly once"

    # e2e: the same batches from pinned host memory through clm_predict_host
    D.barrier()
    t0 = time.perf_counter()
    e2e_pipelined(eng, [(s[1], s[2], s[5][1], s[5][0]) for s in staged], K3_MAX_READS)
    e2e_ms = (time.perf_counter() - t0) * 1e3
    per_rank = D.gather_floats([ms, gather_ms, e2e_ms, my_reads, my_tokens, my_padded, float(loads[D.rank])])
    ms_max = max(r[0] for r in per_rank)
    tokens = [r[4] for r in per_rank]
    real_bases = int(lens.sum())
    return {"workload": f"{'K3' if D.world == 1 else 'K4'}: first {n} reads of the K3 stream (log-normal 1-32 kb, seed {synth.K3_SEED}), "
                        f"length-bucketed into {len(batches)} batches (<= {K3_MAX_READS} reads, <= {K3_TOKEN_CAP} padded tokens), "
                        f"LPT-dealt to {D.world} rank(s), final gather of (index, label)",
            "scaling": "strong", "n_reads": n, "mean_read_len": float(lens.mean()),
            "reads_per_s": n / (ms_max / 1e3), "bases_per_s": real_bases / (ms_max / 1e3),
            "e2e_reads_per_s": n / (max(r[2] for r in per_rank) / 1e3), "e2e_bases_per_s": real_bases / (max(r[2] for r in per_rank) / 1e3),
            "padding_waste": sum(r[5] for r in per_rank) / sum(tokens) - 1.0,
            "ms_per_rank": [r[0] for r in per_rank], "gather_ms_per_rank": [r[1] for r in per_rank],
            "tokens_per_rank": tokens, "reads_per_rank": [r[3] for r in per_rank],
            "token_imbalance_max_over_mean": max(tokens) / (sum(tokens) / len(tokens)),
            "cost_imbalance_max_over_mean": max(r[6] for r in per_rank) / (sum(r[6] for r in per_rank) / len(per_rank)),
            "dense_tensor_frac_of_burst_peak": F_TOK_EXEC * sum(tokens) / D.world / (ms_max / 1e3) / 1e12 / peaks()["tflops_burst"]}


def run_label_agreement(device):
    """Probe-head label agreement against the oracle's golden logits (tests/golden/label_agreement.npz)."""
    from chimeralm_b200.engine import Engine, pack_reads

    from chimeralm_b200.weights import make_state_dict, perturb_norms

    g = np.load(ROOT / "tests" / "golden" / "label_agreement.npz")
    sd = dict(perturb_norms(make_state_dict(0), 1))   # the weights the golden logits were generated with (== tests' state_dict)
    sd["net.head.output_layer.weight"] = torch.from_numpy(g["probe_w"].copy())
    sd["net.head.output_layer.bias"] = torch.from_numpy(g["probe_b"].copy())
    eng = Engine(sd, device=device, max_batch=32, max_tokens=32769, token_budget=12 * 32769)
    logits, labels = [], []
    t0 = time.perf_counter()
    for seqs, _ in synth.label_eval_batches():
        T = max(len(s) for s in seqs) + 1
        bases, offs = pack_reads([s.tobytes() for s in seqs], pinned=True)
        ids, _ = eng.encode(bases, offs, T, **ENC)
        lg, lb = eng.forward(ids, return_labels=True, check=True)
        logits.append(lg.cpu())
        labels.append(lb.cpu())
    dt = time.perf_counter() - t0
    fallbacks = eng.tc_fallbacks
    eng.close()
    got, lab, ref = torch.cat(logits).numpy(), torch.cat(labels).numpy().astype(np.int64), g["logits_probe"]
    margin = ref[:, 1] - ref[:, 0]
    ref_lab = (margin > 0).astype(np.int64)
    return {"label_agreement": float((lab == ref_lab).mean()), "n_reads": int(len(lab)), "n_differ": int((lab != ref_lab).sum()),
            "logit_max_err": float(np.abs(got - ref).max()), "min_abs_oracle_margin": float(np.abs(margin).min()),
            "label1_fraction": float(ref_lab.mean()), "fp32_conv_fallbacks": int(fallbacks),
            "head": "probe (output layer fitted on a calibration draw; every other weight seeded random init) - oracle/make_label_golden.py",
            "reference": "CPU oracle fp32 logits, tests/golden/label_agreement.npz", "seconds": dt}


def run_cli_multi_gpu(world):
    """The mirrored CLI (`python -m chimeralm_b200 predict --gpus N`, one spawned worker per GPU) against a 1-GPU run on
    the same BAM.  Reads of equal length: no padding, so a read's logits do not depend on who shares its batch."""
    from chimeralm_b200.bam import BamWriter, make_record, minimal_header
    from chimeralm_b200.callbacks import load_predictions_from_folder

    tmp = Path(tempfile.mkdtemp(prefix="clm_cli_"))
    bam = tmp / "in.bam"
    seqs, _ = synth.label_reads(96, 31, fixed_len=2000)
    w = BamWriter(bam, minimal_header())
    for i, s in enumerate(seqs):
        w.write(make_record(f"read_{i:04d}", s.tobytes(), sa_tag=True))
    w.close()
    outs = {}
    t0 = time.perf_counter()
    # a clean environment: under torchrun this process carries RANK / WORLD_SIZE / MASTER_* / TORCHELASTIC_* (with
    # TORCHELASTIC_USE_AGENT_STORE the children's own rendezvous would wait on torchrun's store for ever)
    env = {k: v for k, v in os.environ.items()
           if not (k.startswith(("TORCHELASTIC_", "MASTER_", "GROUP_", "ROLE_", "LOCAL_", "NCCL_ASYNC", "TORCH_NCCL_ASYNC"))
                   or k in ("RANK", "WORLD_SIZE", "OMP_NUM_THREADS"))}
    for g in (1, world):
        out = tmp / f"pred{g}"
        try:
            r = subprocess.run([sys.executable, "-m", "chimeralm_b200", "predict", str(bam), "-o", str(out), "-b", "16", "--gpus", str(g)],
                               capture_output=True, text=True, timeout=240, cwd=str(ROOT), env=env)
        except subprocess.TimeoutExpired:
            return {"ok": False, "gpus": g, "error": "timed out after 240 s"}
        if r.returncode != 0:
            return {"ok": False, "gpus": g, "error": (r.stdout + r.stderr)[-400:]}
        outs[g] = load_predictions_from_folder(out)
    files = sorted(p.name for p in (tmp / f"pred{world}").glob("*.txt"))
    return {"ok": outs[1] == outs[world] and len(outs[1]) == 96, "gpus": world, "reads": len(outs[world]),
            "identical_to_single_gpu": outs[1] == outs[world], "rank_files": len(files),
            "ranks_seen": sorted({f.split("_")[0] for f in files}), "seconds": time.perf_counter() - t0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--read-len", type=int, default=READ_LEN)
    ap.add_argument("--cpu-sample", type=int, default=96, help="reads in the CPU baseline sample (0 = skip)")
    ap.add_argument("--k3-reads", type=int, default=24576, help="reads of the K3 stream in the k3 sub-record (0 = skip)")
    ap.add_argument("--k5-steps", type=int, default=16, help="timed K5 batches per GPU (0 = skip)")
    ap.add_argument("--k5-batch", type=int, default=64)
    ap.add_argument("--preheat", type=float, default=1.5, help="seconds of load before the steady-state passes")
    ap.add_argument("--no-labels", action="store_true", help="skip the label-agreement pass")
    ap.add_argument("--no-cli", action="store_true", help="skip the 2-GPU CLI check (only runs at --gpus 2)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's logits and labels as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")

    from chimeralm_b200.config import DEFAULT_CONFIG as cfg
    from chimeralm_b200.weights import make_state_dict

    sd = make_state_dict(0)
    if args.impl == "reference":
        run_reference(args, sd, cfg)
        return

    from chimeralm_b200.engine import Engine

    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    D = Dist(local_rank)
    rank, world = D.rank, D.world
    sampler = ClockSampler(local_rank)   # every rank samples ITS GPU; started now, rows outside the timed regions are dropped
    eng = Engine(sd, device=local_rank, max_batch=args.batch, max_tokens=args.read_len + 1)

    k2 = run_k2(args, eng, D, sampler)
    conv_variant = eng.longconv_variant(k2["T"])

    def guarded(fn, *a):
        # a sub-record must never cost the headline line: its failure is reported in its place.  (Collective calls inside
        # run on every rank or on none - an exception on one rank alone would still hang the others, so only failures
        # that are the same on all ranks, like running out of memory for a shape, are survivable here.)
        try:
            return fn(*a)
        except Exception as e:  # noqa: BLE001
            return {"error": f"{type(e).__name__}: {e}"[:400]}

    k5 = guarded(run_k5, args, eng, D, sampler) if args.k5_steps > 0 else None
    k3 = guarded(run_k3, args, eng, D, sampler) if args.k3_reads > 0 else None
    eng.close()
    D.barrier()
    clocks = sampler.stop()
    ck = clocks.get("k2", {})
    cs = clocks.get("k2_steady", {})
    clocks_per_rank = D.gather_floats([ck.get("sm_mhz") or 0.0, ck.get("sm_mhz_min") or 0.0, ck.get("power_w_max") or 0.0,
                                       float("sw_power_cap" in ck.get("reasons", [])), cs.get("sm_mhz") or 0.0,
                                       cs.get("power_w_max") or 0.0])
    D.close()
    if rank != 0:
        return
    if args.dump_outputs:
        out = Path(args.dump_outputs)
        out.mkdir(parents=True, exist_ok=True)
        for name, t in k2["outputs"].items():
            np.save(out / f"{name}.npy", t.cpu().to(torch.float32).numpy())

    B, L, T, prof = k2["B"], k2["L"], k2["T"], k2["prof"]
    per_rank = k2["per_rank"]   # [ms, gather_ms, ms_profiled, kernel_sum_ms, e2e_ms] per rank
    ms_max = max(r[0] for r in per_rank)
    slow = max(range(world), key=lambda r: per_rank[r][0])
    reads_per_s = world * B * args.steps / (ms_max / 1e3)
    e2e_s = max(r[4] for r in per_rank) / 1e3
    tokens_per_step = B * T
    pk = peaks()
    total_prof_ms = sum(v[0] for v in prof.values())
    # algorithmic work per token per launch (DESIGN.md section 4; SURVEY.md 8(d))
    flop_per_tok = {"gemm_in_proj": 2 * 256 * 768, "gemm_out_proj": 2 * 256 * 256, "gemm_fc1": 2 * 256 * 1024,
                    "gemm_fc2": 2 * 1024 * 256, "block_in": 2 * 256 * 768,
                    "block_mlp": 2 * 256 * 256 + 2 * 256 * 1024 + 2 * 1024 * 256}
    bytes_per_tok = {"longconv": CONV_BYTES_TOK_LAYER, "layernorm": 1024 + 512, "shortconv_gate": 1536 + 1024,
                     "transpose": 1024, "pool": 516, "embed": 1 + 1024 + 512, "encode": 2, "head": 0,
                     "embed_in": 1 + 1024,   # block 0's first half by table lookup: 1 id byte in, x0 + v*x1 (2 x 256 x 2 B) out
                     "gemm_score": 512}   # fused scorer + pooling: the normalised tokens are read once (bf16)
    traffic, traffic_src = {}, None
    for name in ("r2_traffic.json", "r1_traffic.json"):
        tp = ROOT / "profiles" / name
        if tp.exists() and B == BATCH and L == READ_LEN:
            traffic = {k: v for k, v in json.loads(tp.read_text()).items() if not k.startswith("_")}
            traffic_src = f"profiles/{name}: dram__bytes_read.sum + dram__bytes_write.sum per launch from a committed `ncu --set full` capture of this workload (not measured in this run)"
            break

    def roofline_of(name, ms, n):
        sec = ms / n / 1e3
        if name in flop_per_tok:
            ach = flop_per_tok[name] * tokens_per_step / sec / 1e12
            r = {"bound": "tensor", "achieved": ach, "peak": pk["tflops_burst"], "unit": "TFLOP/s", "frac": ach / pk["tflops_burst"],
                 "frac_of_sustained_peak": ach / pk["tflops_sustained"]}
        else:
            ach = bytes_per_tok.get(name, 0) * tokens_per_step / sec / 1e9
            r = {"bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"]}
        r.update({"kernel": name, "traffic": traffic.get(name), "avg_launch_ms": ms / n, "share_of_step": ms / total_prof_ms})
        return r

    dom_name, (dom_ms, dom_n) = max(prof.items(), key=lambda kv: kv[1][0])
    roof = roofline_of(dom_name, dom_ms, dom_n)
    roof["peak_source"] = pk["src"] + ("; burst bf16 figure: the timed region is a fraction of a second, not a power-capped long step"
                                       if roof["bound"] == "tensor" else "")
    roof["traffic_source"] = traffic_src
    rooflines = {k: roofline_of(k, v[0], v[1]) for k, v in prof.items() if k in ("longconv", "block_mlp", "block_in", "gemm_score", "embed_in")}
    if "longconv" in rooflines and conv_variant == "fft_tensor_core":
        # Monarch FFT on tcgen05 (csrc/longconv_tc2.cuh, two items in flight per SM): per item (one channel of two reads) 16
        # MMAs 128x128x16 (step 1) + 2 x 32 MMAs 128x128x16 (steps 3, 5 as N = 128 halves) + 32 MMAs 128x64x16 (step 7; the
        # tail token's row no longer costs an output row); 256 * ceil(B / 2) items per launch.  These are EXECUTED fp16
        # tensor FLOPs (22x the algorithmic FFT count): a pipe-utilisation figure, not a roofline fraction.
        item_flop = 2 * 16 * (16 * 128 * 128 + 2 * 32 * 128 * 128 + 32 * 128 * 64)
        sec = rooflines["longconv"]["avg_launch_ms"] / 1e3
        rooflines["longconv"]["tensor_pipe_executed_tflops"] = item_flop * 256 * ((B + 1) // 2) / sec / 1e12
    dense_tflops = (F_TOK_EXEC if "embed_in" in prof else F_TOK) * (reads_per_s / world) * T / 1e12

    cpu = None
    if args.cpu_sample > 0:
        torch.set_num_threads(os.cpu_count() or 1)
        sample = synth.uniform_reads(args.cpu_sample, L, synth.K2_SEED)
        v, t_tok, t_fwd, _ = cpu_reference_path(sd, cfg, sample)
        cpu = {"value": v, "unit": "reads/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": f"{args.cpu_sample} reads x {L} b of the K2 stream, batch 12 (the reference CLI default); tokenise {t_tok:.2f}s + forward {t_fwd:.2f}s",
               "torch": torch.__version__}
    labels = None if args.no_labels else guarded(run_label_agreement, local_rank)
    cli = guarded(run_cli_multi_gpu, world) if (world == 2 and not args.no_cli) else None

    line = {
        "metric": "predict_reads_per_s", "value": reads_per_s, "unit": "reads/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(L, T, B, world),
        "dtype_note": "bf16 GEMM operands, fp16 operands in the tensor-core FFT conv (power-of-two range scaling, fp32 fallback on overflow), "
                      "fp32 accumulation / residual / pooling / head",
        "bases_per_s": reads_per_s * L,
        "tokens_per_s": reads_per_s * T,
        "dense_tensor_tflops_per_gpu": dense_tflops,
        "dense_tensor_frac_of_burst_peak": dense_tflops / pk["tflops_burst"],
        "dense_tensor_frac_of_sustained_peak": dense_tflops / pk["tflops_sustained"],
        "dense_tensor_note": "executed tensor-core FLOPs only: block 0's in_proj is a lookup over the 16 token ids (embed_in), "
                             "so 393 216 of the graph's 6 423 040 FLOP/token are not counted",
        "e2e": {"value": world * B * args.steps / e2e_s, "unit": "reads/s", "h2d_bytes_per_step": B * L + (B + 1) * 8,
                "d2h_bytes_per_step": B * 2 * 4 + B,
                "api": "clm_predict_host_submit / clm_predict_host_wait (C-ABI, pinned host buffers, up to 3 batches in flight)",
                "one_batch_at_a_time": {"value": world * B * args.steps / (max(r[5] for r in per_rank) / 1e3), "unit": "reads/s",
                                        "api": "clm_predict_host (submit + wait per batch)"}},
        "gpu_launches": int(k2["launches"]),
        "roofline": roof,
        "rooflines_top_kernels": rooflines,
        "longconv_kernel": conv_variant,
        "kernel_ms_per_step": {k: v[0] / args.steps for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])},
        "kernel_ms_per_step_note": "rank 0, from the second (profiled) pass; `value` comes from the first, un-profiled pass",
        "ms_per_rank": [r[0] / args.steps for r in per_rank],
        "compute_ms_per_rank": [(r[0] - r[1]) / args.steps for r in per_rank],   # the same region without the final gather
        "clocks_per_rank": [{"sm_mhz": c[0], "sm_mhz_min": c[1], "power_w_max": c[2], "sw_power_cap": bool(c[3]),
                             "steady_sm_mhz": c[4], "steady_power_w_max": c[5]} for c in clocks_per_rank],
        "gather_ms_per_rank": [r[1] for r in per_rank],
        "slowest_rank": {"rank": slow, "ms_per_step": per_rank[slow][0] / args.steps,
                         "kernel_sum_ms_per_step": per_rank[slow][3] / args.steps,
                         "profiled_pass_ms_per_step": per_rank[slow][2] / args.steps},
        "steady_state": {"value": world * B * args.steps / (max(r[6] for r in per_rank) / 1e3), "unit": "reads/s",
                         "e2e": world * B * args.steps / (max(r[7] for r in per_rank) / 1e3),
                         "ms_per_step": max(r[6] for r in per_rank) / args.steps, "ms_per_rank": [r[6] / args.steps for r in per_rank],
                         "preheat_s": args.preheat, "clocks": clocks.get("k2_steady"),
                         "note": "same K steps after ~1.5 s of the same load: the board is at its power cap; `value` / `e2e` start "
                                 "one second after idle (boost clocks), like round 1's numbers"},
        "label_agreement": labels.get("label_agreement") if labels else None,
        "n_reads": labels.get("n_reads") if labels else None,
        "logit_max_err": labels.get("logit_max_err") if labels else None,
        "labels": labels,
        "k3": k3,
        "k5": k5,
        "cli_multi_gpu": cli,
        "cpu_baseline": cpu,
        "clocks": clocks.get("k2"),
        "clocks_e2e": clocks.get("k2_e2e"),
        "clocks_k3": clocks.get("k3"),
        "clocks_k5": clocks.get("k5"),
    }
    print(json.dumps(line))


if __name__ == "__main__":
    # stdout carries exactly ONE line, the JSON record: libraries that write to fd 1 on their own (NCCL prints its version
    # line there when NCCL_DEBUG is set in the environment) are sent to stderr for the duration of the run
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        import contextlib
        import io

        _buf = io.StringIO()
        with contextlib.redirect_stdout(_buf):
            main()
    finally:
        sys.stdout.flush()
        os.dup2(_real_stdout, 1)
        os.close(_real_stdout)
    sys.stdout.write(_buf.getvalue())
    sys.stdout.flush()
