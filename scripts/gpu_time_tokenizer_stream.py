"""Per-step latency of streaming SoundStream tokenization (SoundStream.stream(...).step) against the offline alternatives,
for the cfg-4 tokenizer (C 256, D 256, K 8192, Euclidean) and the cfg-1 tokenizer (C 256, D 64, K 512, cosine), both on
512 electrodes as in bench.py.  Each round streams 512 bins in 4-bin steps, and at every step the newest tokens are obtained
three ways, each between a pair of CUDA events:

  (a) TokenizerStream.step on the 4 new bins;
  (b) eval get_quantize_vectors on the whole window so far (bins [0, 4t));
  (c) eval get_quantize_vectors on the last 44 bins, the encoder's receptive field: the cheapest exact offline way to get
      the newest token.

The arms alternate within a round, so they share whatever else the machine is doing; the first `--warmup` rounds are
discarded and medians are reported.  The codebook is k-means initialised by one training forward on random data.  A
separate profiled pass (torch.profiler, after the timed rounds) counts the kernels one step of each arm launches at the
last step of the window.  The card's name, power limit and SM clocks are read in the same run.

    python scripts/gpu_time_tokenizer_stream.py --out profiles/r06_tokenizer_stream.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from frankenstein_b200.vq_brain import SoundStream  # noqa: E402

MODELS = {
    "cfg-4": dict(C=256, D=256, codebook_size=8192, n_electrodes=512, use_cosine_sim=False),
    "cfg-1": dict(C=256, D=64, codebook_size=512, n_electrodes=512, use_cosine_sim=True),
}
WINDOW, STEP, FIELD = 512, 4, 44


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    dev = torch.cuda.current_device()
    name, power, clock, max_clock = [s.strip() for s in q[dev].split(",")] if q else (torch.cuda.get_device_name(), "?", "?", "?")
    return {"name": name, "power_limit": power, "sm_clock_at_start": clock, "max_sm_clock": max_clock}


def make_model(cfg):
    torch.manual_seed(0)
    m = SoundStream(**cfg).cuda().train()
    with torch.no_grad():
        m(torch.randn(32, WINDOW, cfg["n_electrodes"], device="cuda"))          # k-means initialisation of the codebook
    return m.eval()


def arms(m, s, x, t):
    """the three ways of getting the tokens of bins [4t - 4, 4t) (t >= 1)"""
    end = STEP * t
    return (lambda: s.step(x[:, end - STEP:end]),
            lambda: m.get_quantize_vectors(x[:, :end]),
            lambda: m.get_quantize_vectors(x[:, max(0, end - FIELD):end]))


@torch.no_grad()
def measure(m, B, rounds, warmup):
    x = torch.randn(B, WINDOW, m.encoder.layers[0].in_channels, device="cuda")
    s = m.stream(B)
    n = WINDOW // STEP
    times = [[[] for _ in range(n)] for _ in range(3)]
    agree_c = agree_b = None
    for r in range(warmup + rounds):
        s.reset()
        ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)] for _ in range(3)]
        outs = [[None] * n for _ in range(3)]
        for t in range(1, n + 1):
            for a, f in enumerate(arms(m, s, x, t)):
                ev[a][t - 1][0].record()
                outs[a][t - 1] = f()
                ev[a][t - 1][1].record()
        torch.cuda.synchronize()
        if r >= warmup:
            for a in range(3):
                for t in range(n):
                    times[a][t].append(ev[a][t][0].elapsed_time(ev[a][t][1]))
        if r == warmup:
            ind = torch.cat([o[0] for o in outs[0]], 1)
            agree_b = (ind == outs[1][-1][0]).float().mean().item()
            newest_c = torch.stack([o[0][:, -1] for o in outs[2]], 1)
            agree_c = (ind == newest_c).float().mean().item()
    med = [[statistics.median(times[a][t]) for t in range(n)] for a in range(3)]
    res = {"batch": B, "rounds": rounds}
    for a, name in enumerate(("a_stream_step", "b_offline_whole_window", "c_offline_last_44_bins")):
        res[name] = {"median_step_ms": round(statistics.median(med[a]), 4),
                     "first_step_ms": round(med[a][0], 4), "last_step_ms": round(med[a][-1], 4),
                     "window_total_ms": round(sum(med[a]), 3),
                     "per_step_ms_at": {str(t): round(med[a][t - 1], 4) for t in (1, 8, 16, 32, 64, 96, 128)}}
    res["index_agreement_stream_vs_b"] = agree_b
    res["index_agreement_stream_vs_c_newest"] = agree_c
    return res


@torch.no_grad()
def launches(m, B):
    """kernels (and memcpy / memset) one step of each arm enqueues at the last step of the window"""
    from torch.profiler import ProfilerActivity, profile
    x = torch.randn(B, WINDOW, m.encoder.layers[0].in_channels, device="cuda")
    s = m.stream(B)
    n = WINDOW // STEP
    for t in range(1, n):
        s.step(x[:, STEP * (t - 1):STEP * t])
    out = {}
    fs = arms(m, s, x, n)
    for f in fs[1:]:
        f()                                         # warm the shapes of the offline arms
    torch.cuda.synchronize()
    for name, f in zip(("a_stream_step", "b_offline_whole_window", "c_offline_last_44_bins"), fs):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            f()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        kinds = {}
        for k in names:
            kinds[k] = kinds.get(k, 0) + 1
        out[name] = {"device_activities": len(names), "by_name": dict(sorted(kinds.items(), key=lambda kv: -kv[1]))}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,32,128")
    ap.add_argument("--models", default="cfg-4,cfg-1")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default="profiles/r06_tokenizer_stream.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures the B200 and has no CPU mode")
    res = {"card": card(), "torch": torch.__version__, "window_bins": WINDOW, "step_bins": STEP, "models": {}}
    for name in a.models.split(","):
        m = make_model(MODELS[name])
        entry = {"config": MODELS[name], "results": []}
        for B in (int(b) for b in a.batches.split(",")):
            entry["results"].append(measure(m, B, a.rounds, a.warmup))
            print(name, json.dumps(entry["results"][-1]), flush=True)
        entry["launches_per_step_batch1"] = launches(m, 1)
        print(name, json.dumps({k: v["device_activities"] for k, v in entry["launches_per_step_batch1"].items()}), flush=True)
        res["models"][name] = entry
        del m
        torch.cuda.empty_cache()
    res["card_at_end"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]), json.dumps(res["card_at_end"]))


if __name__ == "__main__":
    main()
