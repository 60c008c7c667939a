"""Per-step latency of streaming Brainformer encoder inference (Encoder.stream(...).step) against re-running
Encoder.forward on the window so far, at every patch index of the cfg-2 encoder (window 512, patch 32, 256 electrodes,
dim 512, 4 layers, 16 heads x 32).

For each batch size: R rounds, each round one full stream pass (16 one-patch steps, a CUDA event pair around every step)
followed by one offline pass (Encoder.forward on bins [0, 32 t) for t = 1..16, an event pair around each), so the two arms
alternate and share whatever else the machine is doing.  The first `--warmup` rounds are discarded.  Reports the median
per patch index and the largest output difference between the arms.  The card's name, power limit and maximum SM clock
are read in the same run.

    python scripts/gpu_time_stream.py --out profiles/r05_encoder_stream.json
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

CFG2 = dict(window_size=512, n_electrodes=256, patch_size=32, dim=512, n_layers=4, head_dim=32, hidden_dim=2048,
            n_heads=16, n_kv_heads=16)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    dev = torch.cuda.current_device()
    name, power, clock = [s.strip() for s in q[dev].split(",")] if q else (torch.cuda.get_device_name(), "?", "?")
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


@torch.no_grad()
def measure(enc, B, rounds, warmup):
    p, E = enc.patch_size, enc.n_electrodes
    n_patches = enc.n_patches_per_channel
    x = torch.randn(B, enc.config.window_size, E, device="cuda")
    s = enc.stream(B)
    t_stream = [[] for _ in range(n_patches)]
    t_off = [[] for _ in range(n_patches)]
    max_rel = 0.0
    for r in range(warmup + rounds):
        s.reset()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(2 * n_patches)]
        ys = []
        for t in range(n_patches):
            ev[t][0].record()
            ys.append(s.step(x[:, t * p:(t + 1) * p]))
            ev[t][1].record()
        offs = []
        for t in range(n_patches):
            a, b = ev[n_patches + t]
            a.record()
            offs.append(enc(x[:, :(t + 1) * p])[:, -E:])
            b.record()
        torch.cuda.synchronize()
        if r >= warmup:
            for t in range(n_patches):
                t_stream[t].append(ev[t][0].elapsed_time(ev[t][1]))
                t_off[t].append(ev[n_patches + t][0].elapsed_time(ev[n_patches + t][1]))
        if r == warmup:
            for y, o in zip(ys, offs):
                max_rel = max(max_rel, ((y - o).norm() / o.norm()).item())
    rows = []
    for t in range(n_patches):
        ms_s, ms_o = statistics.median(t_stream[t]), statistics.median(t_off[t])
        rows.append({"patch": t + 1, "stream_ms": round(ms_s, 4), "offline_ms": round(ms_o, 4),
                     "stream_ms_min": round(min(t_stream[t]), 4), "offline_ms_min": round(min(t_off[t]), 4),
                     "ratio": round(ms_o / ms_s, 3)})
    total_s, total_o = sum(r_["stream_ms"] for r_ in rows), sum(r_["offline_ms"] for r_ in rows)
    return {"batch": B, "rounds": rounds, "per_patch": rows, "window_stream_ms": round(total_s, 3),
            "window_offline_ms": round(total_o, 3), "max_rel_diff_stream_vs_offline": max_rel}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,32")
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="profiles/r05_encoder_stream.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 and has no CPU mode")
    torch.manual_seed(0)
    enc = bf.Encoder(bf.MAEConfig(**CFG2)).cuda().eval()
    res = {"config": CFG2, "card": card(), "torch": torch.__version__, "results": []}
    for B in (int(b) for b in a.batches.split(",")):
        res["results"].append(measure(enc, B, a.rounds, a.warmup))
        print(json.dumps(res["results"][-1]))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
