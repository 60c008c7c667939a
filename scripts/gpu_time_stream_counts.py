"""Per-step cost of streams whose rows receive different amounts of data in one step (`step(x, counts)`), for the cfg-2
encoder and BrainFormer (window 512, patch 32, 256 electrodes, dim 512, 4 layers, 16 heads x 32; perceiver 32 queries,
2 CrossBlocks) and the cfg-4 tokenizer (C 256, D 256, K 8192, 512 electrodes, 4-bin steps).  Every step feeds one patch
(4 bins for the tokenizer) per row.  At each batch size three arms:

  lockstep   one stream of B rows, `counts=None`: every row takes every step (all rows reset together at the end of the
             window);
  counts     one stream of B rows, seeded counts: each row is idle (count 0) in a step with probability 1/4, otherwise it
             takes the whole step; a row that reaches the end of the window is reset before the next step;
  separate   the same sessions as B batch-1 streams: a stream steps only when its row has data, and is reset with it.

A round is P steps (P = steps per window) of each arm; the arms alternate step by step, so they share whatever else the
machine is doing.  Every step (with its resets) is timed between a pair of CUDA events; the first `--warmup` rounds are
discarded and medians over the remaining steps are reported.  After the timed rounds one step of each arm is profiled
(torch.profiler, CUDA activities): its device activities are counted, and their device time is summed by name for the
lockstep and counts arms.  The card's name, power limit and SM clocks are read in the same run.

    python scripts/gpu_time_stream_counts.py --out profiles/r08_stream_counts.json
"""
import argparse
import json
import os
import random
import statistics
import sys
from collections import defaultdict

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from scripts.gpu_time_stream_sessions import ENC_CFG, PER_CFG, TOK_CFG, TOK_STEP, card, models  # noqa: E402

ARMS = ("lockstep", "counts", "separate")
IDLE = 0.25


class Arms:
    """the three arms of one model at one batch size; plan() draws the next step's resets and counts of the counts arm
    (shared with the separate arm), call(arm, t, plan) enqueues step t"""

    def __init__(self, make, B, bins, P, E, full, seed):
        self.B, self.P, self.full = B, P, full
        self.x = torch.randn(B, bins, E, device="cuda")
        self.lock = make(B)
        self.cnt = make(B)
        self.sep = [make(1) for _ in range(B)]
        self.rng = random.Random(seed)
        self.fed = [0] * B
        self.idle_steps = self.row_steps = 0

    def plan(self):
        resets = [r for r in range(self.B) if self.fed[r] == self.P]
        for r in resets:
            self.fed[r] = 0
        counts = [0 if self.rng.random() < IDLE else self.full for _ in range(self.B)]
        for r in range(self.B):
            self.fed[r] += counts[r] > 0
        self.idle_steps += sum(c == 0 for c in counts)
        self.row_steps += self.B
        return resets, counts

    def call(self, arm, t, plan):
        if arm == "lockstep":
            if t % self.P == 0:
                self.lock.reset()
            return self.lock.step(self.x)
        resets, counts = plan
        if arm == "counts":
            if resets:
                self.cnt.reset(resets)
            return self.cnt.step(self.x, counts)
        for b in resets:
            self.sep[b].reset()
        for b, s in enumerate(self.sep):
            if counts[b]:
                s.step(self.x[b:b + 1])


def device_time_by_name(prof):
    out = defaultdict(float)
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            out[e.name] += e.time_range.elapsed_us()
    return {k: round(v, 2) for k, v in sorted(out.items(), key=lambda kv: -kv[1])}


@torch.no_grad()
def measure(make, bins, P, E, full, B, rounds, warmup, seed):
    a = Arms(make, B, bins, P, E, full, seed)
    times = {k: [] for k in ARMS}
    for r in range(warmup + rounds):
        ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(P)] for k in ARMS}
        for t in range(P):
            plan = a.plan()
            for k in ARMS:
                ev[k][t][0].record()
                a.call(k, t, plan)
                ev[k][t][1].record()
        torch.cuda.synchronize()
        if r >= warmup:
            for k in ARMS:
                times[k] += [s.elapsed_time(e) for s, e in ev[k]]
    res = {"batch": B, "rounds": rounds, "steps_timed": len(times["lockstep"]),
           "idle_row_fraction": round(a.idle_steps / a.row_steps, 4)}
    for k in ARMS:
        res[k] = {"median_step_ms": round(statistics.median(times[k]), 4), "min_step_ms": round(min(times[k]), 4),
                  "max_step_ms": round(max(times[k]), 4)}
    res["counts_over_lockstep"] = round(res["counts"]["median_step_ms"] / res["lockstep"]["median_step_ms"], 3)
    res["separate_over_counts"] = round(res["separate"]["median_step_ms"] / res["counts"]["median_step_ms"], 3)
    # one profiled step of each arm, after the timed rounds (the lockstep arm mid-window)
    from torch.profiler import ProfilerActivity, profile
    plan = a.plan()
    for t in range(P // 2):
        a.call("lockstep", t, None)
    for k in ARMS:
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            a.call(k, P // 2, plan)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        res[k]["device_activities_per_step"] = len(names)
        if k != "separate":
            res[k]["device_us_by_name"] = device_time_by_name(prof)
    del a
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="32,128")
    ap.add_argument("--models", default="cfg-2 encoder,cfg-2 brainformer,cfg-4 tokenizer")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default="profiles/r08_stream_counts.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 and has no CPU mode")
    res = {"card": card(), "torch": torch.__version__, "encoder": ENC_CFG, "perceiver": PER_CFG, "tokenizer": TOK_CFG,
           "tokenizer_step_bins": TOK_STEP, "idle_probability": IDLE, "models": {}}
    ms = models()
    for name in a.models.split(","):
        make, bins, P, E = ms[name]
        full = bins if "tokenizer" in name else 1               # a whole step: bins for the tokenizer, patches otherwise
        res["models"][name] = {"steps_per_window": P, "step_bins": bins, "results": []}
        for B in (int(b) for b in a.batches.split(",")):
            r = measure(make, bins, P, E, full, B, a.rounds, a.warmup, a.seed + B)
            res["models"][name]["results"].append(r)
            print(name, json.dumps({k: v for k, v in r.items() if k not in ARMS}),
                  {k: r[k]["median_step_ms"] for k in ARMS}, flush=True)
    res["card_at_end"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]), json.dumps(res["card_at_end"]))


if __name__ == "__main__":
    main()
