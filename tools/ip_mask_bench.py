"""Cost of a regional identity mask (diffusers' ``ip_adapter_masks``) on the cross-attention processor.
Per SD-1.5 attn2 layer shape: the whole processor call (PhotoVerseAttnProcessor2_0.__call__ under no_grad, bf16, K/V
cache on as in the generation loop) with and without a mask, each timed as a CUDA graph of 20 calls over X buffers rotated
through more than L2 (bench._graph_time_us); the two arms alternate `--rounds` times per shape, median reported.  Also the
downsample kernel per query grid, and one `--steps`-step batch-`--batch` generation (run_generation, batched CFG, CUDA graph)
with and without a mask, alternating.
Usage: python tools/ip_mask_bench.py [--rows 16] [--li 1] [--rounds 5] [--out FILE.json]"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from photoverse_b200 import _lib, ops  # noqa: E402
from photoverse_b200.attention_processor import PhotoVerseAttnProcessor2_0  # noqa: E402
from photoverse_b200.host.unet_sd15 import Attention  # noqa: E402


def _layer(C, dev, seed):
    torch.manual_seed(seed)
    attn = Attention(C, 768, 8)
    proc = PhotoVerseAttnProcessor2_0(hidden_size=C, cross_attention_dim=768, num_tokens=(5,))
    attn.set_processor(proc)
    attn.requires_grad_(False).to(device=dev, dtype=torch.bfloat16)
    return attn, proc


def _mask(dev, h=64, w=64):
    m = torch.zeros(1, 1, h, w)
    m[..., : w // 2] = 1.0
    return m.to(dev)


def _event_ms(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=16)
    ap.add_argument("--li", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(1)
    res = {"device": torch.cuda.get_device_name(dev), "rows": a.rows, "li": a.li, "lt": bench.LT, "dtype": "bf16",
           "mask": "binary, 64x64, left half", "shapes": {}, "downsample": {}}
    mask = _mask(dev)
    l2_bytes = 192 << 20
    for (S, C) in sorted(set(bench.LAYER_SHAPES), reverse=True):
        attn, proc = _layer(C, dev, seed=S + C)
        x32 = torch.randn(a.rows, S, C, generator=g)
        nbuf = max(2, min(16, l2_bytes // max(1, 3 * x32.numel() * 2) + 1))
        xs = [x32.to(dev, torch.bfloat16).roll(i, dims=1) for i in range(nbuf)]
        text = torch.randn(a.rows, bench.LT, 768, generator=g).to(dev, torch.bfloat16)
        img = torch.randn(a.rows, a.li, 768, generator=g).to(dev, torch.bfloat16)
        proc.enable_kv_cache(True, static=True)
        arms = {}
        with torch.no_grad():
            proc.prepare_kv(attn, text, img)
            for name, kw in (("unmasked", {}), ("masked", {"ip_adapter_masks": [mask]})):
                y = attn(xs[0], encoder_hidden_states=(text, img), **kw)
                n0 = _lib.launch_count()
                attn(xs[0], encoder_hidden_states=(text, img), **kw)

                def call(i, kw=kw):
                    attn(xs[i], encoder_hidden_states=(text, img), **kw)
                arms[name] = {"call": call, "y": y, "launches": int(_lib.launch_count() - n0), "times": []}
            for _ in range(a.rounds):
                for name in arms:
                    arms[name]["times"].append(bench._graph_time_us(arms[name]["call"], nbuf))
        row = {}
        for name, arm in arms.items():
            row[f"{name}_us"] = round(statistics.median(arm["times"]), 2)
            row[f"{name}_us_all"] = [round(t, 2) for t in arm["times"]]
            row[f"{name}_launches_per_call"] = arm["launches"]
        row["masked_over_unmasked"] = round(row["masked_us"] / row["unmasked_us"], 4)
        res["shapes"][f"S{S}_C{C}"] = row
        print(f"S={S:5d} C={C:5d}  unmasked {row['unmasked_us']:8.2f} us  masked {row['masked_us']:8.2f} us  "
              f"ratio {row['masked_over_unmasked']}  launches {row['unmasked_launches_per_call']}/"
              f"{row['masked_launches_per_call']}", flush=True)
        proc.enable_kv_cache(False)
        del arms, xs
    m32 = mask[:, 0].contiguous()
    for S in (4096, 1024, 256, 64):
        ops.ip_mask_rows(m32, a.rows, S)
        us = _event_ms(lambda: ops.ip_mask_rows(m32, a.rows, S), 200) * 1000
        res["downsample"][f"S{S}"] = {"us": round(us, 2), "note": "eager launches incl. allocation, 200-call mean"}
        print(f"downsample S={S:5d} B={a.rows}: {us:.2f} us", flush=True)
    # one generation with and without the mask
    import photoverse_b200 as pv
    from photoverse_b200.host.pipeline import run_generation, synthetic_inputs
    from photoverse_b200.host.unet_sd15 import UNetSD15
    torch.manual_seed(0)
    unet = UNetSD15()
    pv.set_visual_cross_attention_adapter(unet, num_tokens=(5,))
    ia, ta = pv.PhotoVerseAdapter(num_tokens=5), pv.PhotoVerseAdapter(num_tokens=5)
    for mod in (unet, ia, ta):
        mod.requires_grad_(False).eval().to(device=dev, dtype=torch.bfloat16)
    inp = synthetic_inputs(a.batch, 64, seed=5, device=dev, dtype=torch.bfloat16)
    gen = {"unmasked": [], "masked": []}
    for r in range(a.rounds + 1):
        for name, kw in (("unmasked", {}), ("masked", {"ip_adapter_masks": [mask]})):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run_generation(unet, ia, ta, inp, num_steps=a.steps, guidance_scale=7.5, mode="batched", **kw)
            torch.cuda.synchronize()
            if r > 0:                                       # the first round captures the graphs and warms up
                gen[name].append((time.perf_counter() - t0) * 1000)
    res["generation"] = {"batch": a.batch, "steps": a.steps, "guidance": 7.5, "mode": "batched",
                         "note": "run_generation wall time incl. graph capture and adapters, median over rounds"}
    for name, ts in gen.items():
        res["generation"][f"{name}_ms"] = round(statistics.median(ts), 1)
        res["generation"][f"{name}_ms_all"] = [round(t, 1) for t in ts]
    res["generation"]["masked_over_unmasked"] = round(res["generation"]["masked_ms"] / res["generation"]["unmasked_ms"], 4)
    print("generation", json.dumps({k: v for k, v in res["generation"].items() if not k.endswith("_all")}), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
