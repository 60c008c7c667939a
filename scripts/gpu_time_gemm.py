"""Standalone timing of the library's GEMM kernels at the cfg-4 shapes (M = 128 trials x 4096 tokens) against cuBLAS
(torch.matmul, bf16) on the same operands.  CUDA events, L2 flushed by the operand sizes themselves (>= 0.5 GB).
Usage: python scripts/gpu_time_gemm.py [M]  ->  one JSON line per shape."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from frankenstein_b200 import gemm
from frankenstein_b200.brainformer import build_complex_rope_cache
from frankenstein_b200.ops import RopeSpec


def time_ms(fn, reps=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    M = int(sys.argv[1]) if len(sys.argv) > 1 else 524288
    dev = torch.device("cuda")
    g = torch.Generator(device="cuda").manual_seed(0)

    def rnd(*shape, s=1.0):
        return (torch.randn(*shape, device=dev, generator=g) * s).to(torch.bfloat16)

    x512 = rnd(M, 512)
    rows = []

    def report(name, flops, ours, ref, bytes_min=None):
        t_o, t_r = time_ms(ours), time_ms(ref)
        rec = {"shape": name, "ours_ms": round(t_o, 4), "cublas_ms": round(t_r, 4), "ours_tflops": round(flops / t_o / 1e9, 1),
               "cublas_tflops": round(flops / t_r / 1e9, 1)}
        if bytes_min:
            rec["ours_GBps_alg"] = round(bytes_min / t_o / 1e6, 1)
        rows.append(rec)
        print(json.dumps(rec), flush=True)

    # ---- A-resident NT (K = 512) ----
    for N, nm in ((512, "proj  NT res  N=512  K=512"), (1536, "qkv   NT res  N=1536 K=512")):
        w = rnd(N, 512, s=0.04)
        report(nm, 2.0 * M * N * 512, lambda: gemm.gemm_nt(x512, w), lambda: x512 @ w.t(), M * (512 + N) * 2)
    w = rnd(1536, 512, s=0.04)
    spec = RopeSpec.from_complex(build_complex_rope_cache(32, 4096, 10000.0).to(dev), 4096, last=True)
    report("qkv+rope  NT res  N=1536 K=512", 2.0 * M * 1536 * 512,
           lambda: gemm.gemm_nt(x512, w, None, gemm.EPI_ROPE, rope=spec, rope_cols=1024, rope_S=4096), lambda: x512 @ w.t(),
           M * (512 + 1536) * 2)
    w13 = rnd(4096, 512, s=0.04)
    report("w13+swiglu NT res N=4096 K=512", 2.0 * M * 4096 * 512, lambda: gemm.gemm_nt(x512, w13, None, gemm.EPI_SWIGLU),
           lambda: x512 @ w13.t(), M * (512 + 4096 + 2048) * 2)
    h13, gated = gemm.gemm_nt(x512, w13, None, gemm.EPI_SWIGLU)
    # ---- streaming NT ----
    w2 = rnd(512, 2048, s=0.02)
    report("w2    NT stream N=512 K=2048", 2.0 * M * 512 * 2048, lambda: gemm.gemm_nt(gated, w2), lambda: gated @ w2.t(),
           M * (2048 + 512) * 2)
    w13t = rnd(512, 4096, s=0.02)
    report("w13dx NT stream N=512 K=4096", 2.0 * M * 512 * 4096, lambda: gemm.gemm_nt(h13, w13t), lambda: h13 @ w13t.t(),
           M * (4096 + 512) * 2)
    qkv = rnd(M, 1536)
    wqt = rnd(512, 1536, s=0.02)
    report("qkvdx NT stream N=512 K=1536", 2.0 * M * 512 * 1536, lambda: gemm.gemm_nt(qkv, wqt), lambda: qkv @ wqt.t(),
           M * (1536 + 512) * 2)
    # ---- TN ----
    report("w13dw TN 4096x512", 2.0 * M * 4096 * 512, lambda: gemm.gemm_tn(h13, x512), lambda: h13.t() @ x512, M * (4096 + 512) * 2)
    report("w2dw  TN 512x2048", 2.0 * M * 512 * 2048, lambda: gemm.gemm_tn(x512, gated), lambda: x512.t() @ gated, M * (2048 + 512) * 2)
    report("qkvdw TN 1536x512", 2.0 * M * 1536 * 512, lambda: gemm.gemm_tn(qkv, x512), lambda: qkv.t() @ x512, M * (1536 + 512) * 2)
    report("projdw TN 512x512", 2.0 * M * 512 * 512, lambda: gemm.gemm_tn(x512, x512), lambda: x512.t() @ x512, M * 1024 * 2)


if __name__ == "__main__":
    main()
