"""Head_dim 16, 32 and 64 at the same inner width (512), one JSON line on stdout (and to --out).

* attention forward + backward, 16 trials x 4096 tokens, block-causal with 256 electrodes, arms alternated per rep:
  (a) 16 x 32 on the head_dim-32 tcgen05 kernels, (b) 8 x 64 on the head_dim-64 tcgen05 kernels, (c) 8 x 64 through
  library SDPA with the dense [B,1,S,S] bool mask (the only way head_dim 64 ran before), (d) 32 x 16 on the head_dim-16
  instantiation of the tcgen05 kernels, (e) 32 x 16 through library SDPA with the dense mask.  Per-kernel ms from CUDA
  events (_lib.TIMER), algorithmic TF/s = the visible-pair flop count of bench.py (forward 2, backward 5 score-shaped
  matmuls).  Each rep runs on a fresh qkv buffer of 201 MB (> the 126 MB L2).
* train-step trials/s of the cfg-2 BrainFormer (bench.py ENC_CFG / PER_CFG, 128 trials, bf16 autocast, AdamW + value
  clip) with the encoder heads of each selected tcgen05 arm.

Usage: python scripts/gpu_time_head_dim.py [--reps 7] [--arms a,b,c,d,e] [--out result.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

from frankenstein_b200 import _lib, ops

B, S, E, INNER = 16, 4096, 256, 512


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def elapsed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def attention_arms(reps, selected):
    dev = torch.device("cuda")
    mask = ops.LabelMask.block_causal(B, S, E, dev)
    pairs = float(mask.visible_pairs())
    dense = mask.dense()
    g = torch.Generator(device=dev).manual_seed(0)
    w = torch.randn(B, S, INNER, device=dev, generator=g).to(torch.bfloat16)

    def ours(hd):
        H = INNER // hd

        def run():
            x = (torch.randn(B, S, 3 * INNER, device=dev, generator=g) * 1.2).to(torch.bfloat16).requires_grad_(True)
            torch.cuda.synchronize()
            _lib.TIMER.reset()
            _lib.TIMER.enabled = True
            t = elapsed(lambda: ops.attention_qkv(x * 1.0, H, None, mask).backward(w))
            _lib.TIMER.enabled = False
            return t, {k: v[1] for k, v in _lib.TIMER.summary().items()}
        return run

    def sdpa(hd):
        H = INNER // hd

        def run():
            x = (torch.randn(B, S, 3 * INNER, device=dev, generator=g) * 1.2).to(torch.bfloat16).requires_grad_(True)
            torch.cuda.synchronize()

            def body():
                q, k, v = x.view(B, S, 3, H, hd).unbind(2)
                o = F.scaled_dot_product_attention(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2), attn_mask=dense)
                o.transpose(1, 2).reshape(B, S, INNER).backward(w)
            return elapsed(body), {}
        return run

    arms = {"a_16x32_tc": ours(32), "b_8x64_tc": ours(64), "c_8x64_sdpa_dense": sdpa(64), "d_32x16_tc": ours(16),
            "e_32x16_sdpa_dense": sdpa(16)}
    arms = {k: v for k, v in arms.items() if k[0] in selected}
    for fn in arms.values():          # warm-up of every shape
        fn(); fn()
    times = {k: [] for k in arms}
    kern = {k: {} for k in arms}
    for _ in range(reps):
        for name, fn in arms.items():
            t, ks = fn()
            times[name].append(t)
            for kk, ms in ks.items():
                kern[name].setdefault(kk, []).append(ms)
    flops_f = 2.0 * pairs * 2.0 * INNER               # QK^T and PV over the visible pairs (H * hd = INNER)
    flops_b = 5.0 * pairs * 2.0 * INNER
    out = {}
    for name in arms:
        ms = statistics.median(times[name])
        rec = {"fwd_bwd_ms": round(ms, 3), "alg_tflops": round((flops_f + flops_b) / ms / 1e9, 1),
               "spread_ms": [round(min(times[name]), 3), round(max(times[name]), 3)]}
        for kk, v in kern[name].items():
            km = statistics.median(v)
            work = {"attn_fwd": flops_f, "attn_bwd_dkv": 0.8 * flops_b, "attn_bwd_dq": 0.2 * flops_b}.get(kk)
            rec[kk + "_ms"] = round(km, 3)
            if work:
                rec[kk + "_alg_tflops"] = round(work / km / 1e9, 1)
        out[name] = rec
    return out


def train_steps(reps, selected, trials=128):
    import bench
    from frankenstein_b200.brainformer import BrainFormer, Config, MAEConfig
    dev = torch.device("cuda")
    x, t = bench.synth_batch(trials, 1234)
    x, t = x[..., :256].contiguous().to(dev), t.to(dev)
    models = {}
    heads = {"a": ("16x32", 16, 32), "b": ("8x64", 8, 64), "d": ("32x16", 32, 16)}
    for name, H, hd in (heads[a] for a in "abd" if a in selected):
        enc = dict(bench.ENC_CFG, n_heads=H, n_kv_heads=H, head_dim=hd)
        torch.manual_seed(0)
        m = BrainFormer(Config(encoder=MAEConfig(**enc), **bench.PER_CFG)).to(dev).train()
        params = [p for p in m.parameters() if p.requires_grad]
        opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=0.01, fused=True)

        def step(m=m, opt=opt, params=params):
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                loss = m(x, t)[0]
            loss.backward()
            torch.nn.utils.clip_grad_value_(params, 1.0)
            opt.step()
            return loss
        models[name] = step
    for step in models.values():
        for _ in range(3):
            step()
    torch.cuda.synchronize()
    res = {k: [] for k in models}
    for _ in range(reps):
        for name, step in models.items():
            ms = elapsed(lambda: [step() for _ in range(4)]) / 4
            res[name].append(trials / (ms / 1e3))
    return {k: {"trials_per_s": round(statistics.median(v), 1), "spread": [round(min(v), 1), round(max(v), 1)]}
            for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--arms", default="a,b,c,d,e", help="comma-separated attention arms (train steps: a, b, d among them)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    selected = set(args.arms.split(","))
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: these are GPU timings")
    rec = {"gpu": gpu_info(), "shape": f"{B} trials x {S} tokens, block-causal E={E}, inner width {INNER}",
           "attention": attention_arms(args.reps, selected),
           "train_step_cfg2": train_steps(max(3, args.reps // 2), selected)}
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
