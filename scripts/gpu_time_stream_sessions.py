"""Per-step cost of streams whose batch rows are independent sessions, for the cfg-2 encoder and BrainFormer (window 512,
patch 32, 256 electrodes, dim 512, 4 layers, 16 heads x 32; perceiver 32 queries, 2 CrossBlocks) and the cfg-4 tokenizer
(C 256, D 256, K 8192, 512 electrodes, 4-bin steps).  At each batch size three arms feed the same number of sessions:

  lockstep   one stream of B rows, every row at the same position (reset together at the end of the window);
  staggered  one stream of B rows at different positions: before step t the rows r with (r + t) % P == 0 are reset, so
             every row restarts every P steps (P = steps per window) and the resets are spread over the steps;
  separate   B batch-1 streams, one step of each per step (the only way to run unsynchronised sessions without per-row
             state).

A round is P steps of each arm; the arms alternate step by step, so they share whatever else the machine is doing.  Every
step (with its resets) is timed between a pair of CUDA events; the first `--warmup` rounds are discarded and medians over
the remaining steps are reported.  One profiled step of each arm (torch.profiler, after the timed rounds) counts its device
activities (kernels, memsets, copies).  The card's name, power limit and SM clocks are read in the same run.

    python scripts/gpu_time_stream_sessions.py --out profiles/r07_stream_sessions.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from frankenstein_b200 import brainformer as bf  # noqa: E402
from frankenstein_b200.vq_brain import SoundStream  # noqa: E402

ENC_CFG = dict(window_size=512, n_electrodes=256, patch_size=32, dim=512, n_layers=4, head_dim=32, hidden_dim=2048,
               n_heads=16, n_kv_heads=16)
PER_CFG = dict(n_output_tokens=32, output_dim=768, dim=512, n_layers=2, head_dim=16, hidden_dim=512, n_heads=4, n_kv_heads=4)
TOK_CFG = dict(C=256, D=256, codebook_size=8192, n_electrodes=512, use_cosine_sim=False)
TOK_STEP, TOK_STEPS = 4, 16                     # the tokenizer's window here: 16 steps of 4 bins


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    dev = torch.cuda.current_device()
    name, power, clock, max_clock = [s.strip() for s in q[dev].split(",")] if q else (torch.cuda.get_device_name(), "?", "?", "?")
    return {"name": name, "power_limit": power, "sm_clock_at_start": clock, "max_sm_clock": max_clock}


def models():
    torch.manual_seed(0)
    enc = bf.Encoder(bf.MAEConfig(**ENC_CFG)).cuda().eval()
    torch.manual_seed(0)
    bfm = bf.BrainFormer(bf.Config(encoder=bf.MAEConfig(**ENC_CFG), **PER_CFG)).cuda().eval()
    torch.manual_seed(0)
    tok = SoundStream(**TOK_CFG).cuda().train()
    with torch.no_grad():
        tok(torch.randn(32, 512, TOK_CFG["n_electrodes"], device="cuda"))         # k-means initialisation of the codebook
    tok.eval()
    p = ENC_CFG["patch_size"]
    n_enc = ENC_CFG["window_size"] // p
    return {"cfg-2 encoder": (lambda B: enc.stream(B), p, n_enc, ENC_CFG["n_electrodes"]),
            "cfg-2 brainformer": (lambda B: bfm.stream(B), p, n_enc, ENC_CFG["n_electrodes"]),
            "cfg-4 tokenizer": (lambda B: tok.stream(B), TOK_STEP, TOK_STEPS, TOK_CFG["n_electrodes"])}


class Arms:
    """the three arms of one model at one batch size; call(arm, t) enqueues step t of the window (t = 0 .. P - 1)"""

    def __init__(self, make, B, bins, P, E):
        self.B, self.bins, self.P = B, bins, P
        self.x = torch.randn(B, bins, E, device="cuda")
        self.lock = make(B)
        self.stag = make(B)
        self.sep = [make(1) for _ in range(B)]

    def call(self, arm, t):
        x = self.x
        if arm == "lockstep":
            if t == 0:
                self.lock.reset()
            return self.lock.step(x)
        if arm == "staggered":
            rows = [r for r in range(self.B) if (r + t) % self.P == 0]
            if rows:
                self.stag.reset(rows)
            return self.stag.step(x)
        for b, s in enumerate(self.sep):
            if t == 0:
                s.reset()
            s.step(x[b:b + 1])

    def prime(self):
        """bring the staggered stream to its steady state (every row mid-session) without timing"""
        for t in range(self.P):
            self.call("staggered", t)


ARMS = ("lockstep", "staggered", "separate")


@torch.no_grad()
def measure(make, bins, P, E, B, rounds, warmup):
    a = Arms(make, B, bins, P, E)
    a.prime()
    times = {k: [] for k in ARMS}
    for r in range(warmup + rounds):
        ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(P)] for k in ARMS}
        for t in range(P):
            for k in ARMS:
                ev[k][t][0].record()
                a.call(k, t)
                ev[k][t][1].record()
        torch.cuda.synchronize()
        if r >= warmup:
            for k in ARMS:
                times[k] += [s.elapsed_time(e) for s, e in ev[k]]
    res = {"batch": B, "rounds": rounds, "steps_timed": len(times["lockstep"])}
    for k in ARMS:
        res[k] = {"median_step_ms": round(statistics.median(times[k]), 4), "min_step_ms": round(min(times[k]), 4),
                  "max_step_ms": round(max(times[k]), 4)}
    res["staggered_over_lockstep"] = round(res["staggered"]["median_step_ms"] / res["lockstep"]["median_step_ms"], 3)
    res["separate_over_staggered"] = round(res["separate"]["median_step_ms"] / res["staggered"]["median_step_ms"], 3)
    # device activities of one step of each arm, mid-window (t = P // 2: the staggered arm resets rows at most steps)
    from torch.profiler import ProfilerActivity, profile
    t = P // 2
    for k in ARMS:
        for u in range(t):
            a.call(k, u)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            a.call(k, t)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        res[k]["device_activities_per_step"] = len(names)
    del a
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,32,128")
    ap.add_argument("--models", default="cfg-2 encoder,cfg-2 brainformer,cfg-4 tokenizer")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default="profiles/r07_stream_sessions.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 and has no CPU mode")
    res = {"card": card(), "torch": torch.__version__, "encoder": ENC_CFG, "perceiver": PER_CFG, "tokenizer": TOK_CFG,
           "tokenizer_step_bins": TOK_STEP, "models": {}}
    ms = models()
    for name in a.models.split(","):
        make, bins, P, E = ms[name]
        res["models"][name] = {"steps_per_window": P, "step_bins": bins, "results": []}
        for B in (int(b) for b in a.batches.split(",")):
            r = measure(make, bins, P, E, B, a.rounds, a.warmup)
            res["models"][name]["results"].append(r)
            print(name, json.dumps(r), flush=True)
    res["card_at_end"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]), json.dumps(res["card_at_end"]))


if __name__ == "__main__":
    main()
