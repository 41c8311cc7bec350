"""Whole cross-attention processor call (PhotoVerseAttnProcessor2_0.__call__ under no_grad, K/V cache on as in the
generation loop) per SD-1.5 attn2 layer shape, float16 model against bfloat16 model on the same weights and inputs.
Each call is timed as a CUDA graph of 20 calls over X buffers rotated through more than L2 (bench._graph_time_us);
the two dtypes alternate `--rounds` times per shape and the median per dtype is reported.
Usage: python tools/f16_bench.py [--rows 16] [--li 1] [--rounds 5] [--out FILE.json]"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from photoverse_b200 import _lib  # noqa: E402
from photoverse_b200.attention_processor import PhotoVerseAttnProcessor2_0  # noqa: E402
from photoverse_b200.host.unet_sd15 import Attention  # noqa: E402

DTYPES = {"bf16": torch.bfloat16, "f16": torch.float16}


def _layer(C, dev, seed):
    torch.manual_seed(seed)
    attn = Attention(C, 768, 8)
    proc = PhotoVerseAttnProcessor2_0(hidden_size=C, cross_attention_dim=768, num_tokens=(5,))
    attn.set_processor(proc)
    attn.requires_grad_(False).to(dev)
    return attn, proc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=16)
    ap.add_argument("--li", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(1)
    res = {"device": torch.cuda.get_device_name(dev), "rows": a.rows, "li": a.li, "lt": bench.LT, "shapes": {}}
    l2_bytes = 192 << 20
    for (S, C) in sorted(set(bench.LAYER_SHAPES), reverse=True):
        x32 = torch.randn(a.rows, S, C, generator=g)
        text32 = torch.randn(a.rows, bench.LT, 768, generator=g)
        img32 = torch.randn(a.rows, a.li, 768, generator=g)
        nbuf = max(2, min(16, l2_bytes // max(1, 3 * x32.numel() * 2) + 1))
        arms = {}
        for name, dt in DTYPES.items():
            attn, proc = _layer(C, dev, seed=S + C)          # identical fp32 masters in both arms
            xs = [x32.to(dev, dt).roll(i, dims=1) for i in range(nbuf)]
            text, img = text32.to(dev, dt), img32.to(dev, dt)
            proc.enable_kv_cache(True, static=True)
            with torch.no_grad():
                proc.prepare_kv(attn, text, img)
                y = attn(xs[0], encoder_hidden_states=(text, img))
                n0 = _lib.launch_count()
                attn(xs[0], encoder_hidden_states=(text, img))
                launches = int(_lib.launch_count() - n0)

                def call(i, attn=attn, xs=xs, text=text, img=img):
                    attn(xs[i], encoder_hidden_states=(text, img))
            arms[name] = {"call": call, "y": y, "launches": launches, "times": [], "keep": (attn, proc, xs, text, img)}
        for _ in range(a.rounds):
            for name in DTYPES:                                # alternate the two builds of the layer
                with torch.no_grad():
                    arms[name]["times"].append(bench._graph_time_us(arms[name]["call"], nbuf))
        row = {}
        for name in DTYPES:
            row[f"{name}_us"] = round(statistics.median(arms[name]["times"]), 2)
            row[f"{name}_us_all"] = [round(t, 2) for t in arms[name]["times"]]
            row[f"{name}_launches_per_call"] = arms[name]["launches"]
        row["f16_over_bf16"] = round(row["f16_us"] / row["bf16_us"], 3)
        row["max_abs_f16_vs_bf16"] = float((arms["f16"]["y"].float() - arms["bf16"]["y"].float()).abs().max())
        res["shapes"][f"S{S}_C{C}"] = row
        print(f"S={S:5d} C={C:5d}  bf16 {row['bf16_us']:8.2f} us  f16 {row['f16_us']:8.2f} us  ratio {row['f16_over_bf16']}"
              f"  launches {row['bf16_launches_per_call']}/{row['f16_launches_per_call']}", flush=True)
        for arm in arms.values():
            arm["keep"][1].enable_kv_cache(False)
        del arms
        torch.cuda.empty_cache()
    tot = {n: sum(res["shapes"][f"S{S}_C{C}"][f"{n}_us"] for S, C in bench.LAYER_SHAPES) for n in DTYPES}
    res["unet_eval_16_layers_us"] = {n: round(t, 1) for n, t in tot.items()}
    print(json.dumps(res["unet_eval_16_layers_us"]))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
