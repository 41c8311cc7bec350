"""GEGLU feed-forward projection timing at the transformer-block shapes of a batch-8 (16-row) latent-64 generation:
F.linear + ops.geglu (two launches, the [M, 2N] projection goes through HBM) against ops.linear_geglu (one launch), and
the plain persistent CTA-pair GEMM (ops.linear) at the same [M, K] x [2N, K] shape, so that GEMM speed and epilogue cost
can be told apart.  CUDA graph of 20 launches (bench.py:_graph_time_us) over buffers rotated beyond the 126 MB L2.

    python tools/geglu_bench.py [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import _graph_time_us, measured_peaks  # noqa: E402
from photoverse_b200 import ops  # noqa: E402

# (M, C): ff.proj of the transformer blocks at 16 rows, S = 4096 / 1024 / 256 / 64 (mid block)
SHAPES = [(65536, 320), (16384, 640), (4096, 1280), (1024, 1280)]
ROTATE_BYTES = 512 << 20


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                      # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    dt = torch.bfloat16
    peaks = measured_peaks()
    info = gpu_info()
    print(json.dumps({"gpu": info, "peaks": peaks}))
    rows = []
    g = torch.Generator().manual_seed(5)
    for M, C in SHAPES:
        K, N = C, 4 * C
        per_set = 2 * (M * K + M * 2 * N + M * N)
        nbuf = max(2, min(64, -(-ROTATE_BYTES // per_set)))
        x = [torch.randn(M, K, generator=g).to(dev, dt) for _ in range(nbuf)]
        lin = torch.nn.Linear(K, 2 * N).to(dev, dt)
        w, b = lin.weight.detach(), lin.bias.detach()
        wp, bp = ops.pack_geglu_weight(w, b)
        b32 = b.float()
        h = [torch.empty(M, 2 * N, device=dev, dtype=dt) for _ in range(nbuf)]
        y = [torch.empty(M, N, device=dev, dtype=dt) for _ in range(nbuf)]

        def unfused(i):
            ops.geglu(F.linear(x[i], w, b))

        def fused(i):
            ops.linear_geglu(x[i], wp, bp)

        def gemm(i):
            ops.linear(x[i], w, b32, out=h[i])

        with torch.no_grad():
            ref = ops.geglu(F.linear(x[0], w, b))
            out = ops.linear_geglu(x[0], wp, bp)
            d = (ref.float() - out.float()).abs()
            t_unf = _graph_time_us(unfused, nbuf)
            t_fus = _graph_time_us(fused, nbuf)
            t_gemm = _graph_time_us(gemm, nbuf)
        flops = 2.0 * M * (2 * N) * K
        r = {"M": M, "K": K, "N": N, "nbuf": nbuf,
             "unfused_us": round(t_unf, 1), "fused_us": round(t_fus, 1), "gemm3_us": round(t_gemm, 1),
             "fused_over_unfused": round(t_fus / t_unf, 3),
             "fused_tflops": round(flops / t_fus / 1e6, 1), "gemm3_tflops": round(flops / t_gemm / 1e6, 1),
             "unfused_tflops": round(flops / t_unf / 1e6, 1),
             "fused_share_of_peak": round(flops / t_fus / 1e6 / peaks["bf16_tflops"], 3),
             "max_abs_diff_vs_unfused": float(d.max()), "frac_equal": float((d == 0).float().mean())}
        rows.append(r)
        print(json.dumps(r), flush=True)
        del x, h, y
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"gpu": info, "peaks": peaks, "shapes": rows}, f, indent=1)


if __name__ == "__main__":
    main()
