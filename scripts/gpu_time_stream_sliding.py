"""Per-step cost of sliding streams (`stream(B, sliding=True)`) over sessions longer than the window, for the cfg-2 encoder
and BrainFormer (window 512, patch 32, 256 electrodes, dim 512, 4 layers, 16 heads x 32; perceiver 32 queries,
2 CrossBlocks).  Every step feeds one patch per row; a session runs 4 windows (4 W = 64 steps).  At each batch size three
arms:

  sliding   one sliding stream of B rows, stepped through the 4 windows;
  bounded   one bounded stream of B rows (`sliding=False`) in lockstep over the first window only, reset at its end;
  forward   `forward` re-run on the last W patches (fewer at the start) at each step, the cost a sliding stream avoids.

A round is 4 W steps of each arm; the arms alternate step by step, so they share whatever else the machine is doing.
Every step is timed between a pair of CUDA events; the first `--warmup` rounds are discarded (they also warm every shape
of the forward arm) and medians over the remaining steps are reported.  The sliding arm is reported per window: its
median over windows 2-4 against its median over window 1 shows whether its cost grows with the session's length.  The
kernel device time inside a step is not measured here.  The card's name, power limit and SM clocks are read in the same
run.

    python scripts/gpu_time_stream_sliding.py --out profiles/r09_stream_sliding.json
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from frankenstein_b200 import brainformer as bf  # noqa: E402
from scripts.gpu_time_stream_sessions import ENC_CFG, PER_CFG, card  # noqa: E402

ARMS = ("sliding", "bounded", "forward")
WINDOWS = 4


def models():
    torch.manual_seed(0)
    enc = bf.Encoder(bf.MAEConfig(**ENC_CFG)).cuda().eval()
    torch.manual_seed(0)
    bfm = bf.BrainFormer(bf.Config(encoder=bf.MAEConfig(**ENC_CFG), **PER_CFG)).cuda().eval()
    return {"cfg-2 encoder": (enc, lambda B, sliding: enc.stream(B, sliding=sliding), lambda x: enc(x)),
            "cfg-2 brainformer": (enc, lambda B, sliding: bfm.stream(B, sliding=sliding), lambda x: bfm(x)[1])}


@torch.no_grad()
def measure(enc, make, fwd, B, rounds, warmup, seed):
    p, E, W = enc.patch_size, enc.n_electrodes, enc.n_patches_per_channel
    n = WINDOWS * W
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, n * p, E, device="cuda", generator=g)
    times = {k: [[] for _ in range(n)] for k in ARMS}
    for r in range(warmup + rounds):
        sl, bd = make(B, True), make(B, False)
        ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)] for k in ARMS}
        for t in range(n):
            for k in ARMS:
                ev[k][t][0].record()
                if k == "sliding":
                    sl.step(x[:, t * p:(t + 1) * p])
                elif k == "bounded":
                    if t % W == 0:
                        bd.reset()
                    bd.step(x[:, (t % W) * p:(t % W + 1) * p])
                else:
                    fwd(x[:, max(0, t + 1 - W) * p:(t + 1) * p])
                ev[k][t][1].record()
        torch.cuda.synchronize()
        if r >= warmup:
            for k in ARMS:
                for t, (s, e) in enumerate(ev[k]):
                    times[k][t].append(s.elapsed_time(e))
        assert sl.lengths == [n * E] * B
        del sl, bd
    med = lambda ts: round(statistics.median(ts), 4)  # noqa: E731
    flat = lambda k, lo, hi: [v for t in range(lo, hi) for v in times[k][t]]  # noqa: E731
    res = {"batch": B, "rounds": rounds, "steps_timed_per_arm": rounds * n}
    res["sliding"] = {f"window_{w + 1}_median_step_ms": med(flat("sliding", w * W, (w + 1) * W)) for w in range(WINDOWS)}
    res["sliding"]["windows_2_4_median_step_ms"] = med(flat("sliding", W, n))
    res["sliding"]["median_step_ms"] = med(flat("sliding", 0, n))
    res["bounded"] = {"median_step_ms": med(flat("bounded", 0, n))}
    res["forward"] = {"median_step_ms": med(flat("forward", 0, n)), "full_window_median_step_ms": med(flat("forward", W - 1, n))}
    s = res["sliding"]
    res["sliding_windows_2_4_over_window_1"] = round(s["windows_2_4_median_step_ms"] / s["window_1_median_step_ms"], 3)
    res["sliding_over_bounded"] = round(s["median_step_ms"] / res["bounded"]["median_step_ms"], 3)
    res["forward_over_sliding"] = round(res["forward"]["median_step_ms"] / s["median_step_ms"], 3)
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,32,128")
    ap.add_argument("--models", default="cfg-2 encoder,cfg-2 brainformer")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default="profiles/r09_stream_sliding.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 and has no CPU mode")
    res = {"card": card(), "torch": torch.__version__, "encoder": ENC_CFG, "perceiver": PER_CFG, "windows": WINDOWS,
           "kernel_device_time_in_step": "not measured", "models": {}}
    ms = models()
    for name in a.models.split(","):
        enc, make, fwd = ms[name]
        res["models"][name] = {"steps_per_window": enc.n_patches_per_channel, "results": []}
        for B in (int(b) for b in a.batches.split(",")):
            r = measure(enc, make, fwd, B, a.rounds, a.warmup, a.seed + B)
            res["models"][name]["results"].append(r)
            print(name, json.dumps(r), flush=True)
    res["card_at_end"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]), json.dumps(res["card_at_end"]))


if __name__ == "__main__":
    main()
