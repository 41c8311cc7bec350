"""float32 models under torch.autocast (DESIGN.md 4.9): what the conversions cost and what the 16-bit path saves.

  * pv_convert_fwd bandwidth, fp32 -> bf16 and bf16 -> fp32, over buffers larger than L2, against a 6.5 TB/s copy peak;
  * the whole processor call (no_grad, static K/V cache as in the generation loop) per SD-1.5 attn2 layer shape in four arms
    on the same fp32 masters, each timed as a CUDA graph of 20 calls over X buffers rotated through more than L2
    (bench._graph_time_us), the arms alternating `--rounds` times, median per arm:
        bf16          a bf16 model (bf16 X, text and image tokens)
        ac_bf16_x     a float32 model under bf16 autocast with bf16 X (this repo's host UNet: its LayerNorm kernel emits bf16),
                      float32 text states and bf16 image tokens
        ac_f32_x      the same with float32 X (diffusers: nn.LayerNorm returns float32 under autocast): X conversion included
        f32           a float32 model without autocast (the fp32 SIMT parity path)
    plus the conversion of X alone (convert_x_us);
  * the training step (ms) of a float32 UNet under bf16 autocast next to bench.py's training configuration (bf16 backbone,
    float32 masters of the trainable set), batch `--train-batch`, latent 64^2, LoRA r = 8, CLIP text tower.
Usage: python tools/autocast_bench.py [--rows 16] [--li 1] [--rounds 5] [--train-batch 16] [--out FILE.json]"""
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

BF16, F32 = torch.bfloat16, torch.float32
COPY_PEAK_GBS = 6500.0
ARMS = ("bf16", "ac_bf16_x", "ac_f32_x", "f32")


def _autocast(on):
    return torch.autocast("cuda", dtype=BF16, enabled=on, cache_enabled=False)


def convert_bandwidth(dev):
    n = 64 << 20                                   # 256 MB of fp32, 128 MB of bf16: both beyond the 126 MB of L2
    x32 = torch.randn(n, device=dev)
    x16 = x32.to(BF16)
    out = {}
    for name, src, dt in (("f32_to_bf16", x32, BF16), ("bf16_to_f32", x16, F32)):
        for _ in range(3):
            ops.convert(src, dt)
        torch.cuda.synchronize()
        times = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                ops.convert(src, dt)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1) / 10 * 1e3)
        us = statistics.median(times)
        gbs = n * 6 / (us * 1e-6) / 1e9
        out[name] = {"elements": n, "bytes_moved": n * 6, "us": round(us, 1), "GB_per_s": round(gbs, 1),
                     "fraction_of_6.5TBps_copy_peak": round(gbs / COPY_PEAK_GBS, 3)}
        print(f"{name}: {us:.1f} us, {gbs:.0f} GB/s ({gbs / COPY_PEAK_GBS:.1%} of {COPY_PEAK_GBS:.0f} GB/s)", flush=True)
    return out


def _layer(C, dev, seed, dtype):
    torch.manual_seed(seed)
    attn = Attention(C, 768, 8)
    proc = PhotoVerseAttnProcessor2_0(hidden_size=C, cross_attention_dim=768, num_tokens=(5,))
    attn.set_processor(proc)
    attn.requires_grad_(False).to(dev, dtype)
    return attn, proc


def layer_times(dev, rows, li, rounds):
    g = torch.Generator().manual_seed(1)
    shapes = {}
    l2_bytes = 192 << 20
    for (S, C) in sorted(set(bench.LAYER_SHAPES), reverse=True):
        x32 = torch.randn(rows, S, C, generator=g)
        text32 = torch.randn(rows, bench.LT, 768, generator=g).to(dev)
        img32 = torch.randn(rows, li, 768, generator=g).to(dev)
        nbuf = max(2, min(16, l2_bytes // max(1, 3 * x32.numel() * 2) + 1))
        spec = {"bf16": (BF16, BF16, BF16, False), "ac_bf16_x": (F32, BF16, F32, True),
                "ac_f32_x": (F32, F32, F32, True), "f32": (F32, F32, F32, False)}   # model, X, text dtypes; autocast
        arms = {}
        for name, (mdt, xdt, tdt, ac) in spec.items():
            attn, proc = _layer(C, dev, S + C, mdt)        # identical fp32 masters in every arm
            xs = [x32.to(dev, xdt).roll(i, dims=1) for i in range(nbuf)]
            text = text32.to(tdt)
            img = img32.to(BF16 if ac else mdt)             # under autocast the adapter hands over bf16 tokens
            proc.enable_kv_cache(True, static=True)
            with torch.no_grad(), _autocast(ac):
                proc.prepare_kv(attn, text, img)
                y = attn(xs[0], encoder_hidden_states=(text, img))
                n0 = _lib.launch_count()
                attn(xs[0], encoder_hidden_states=(text, img))
                launches = int(_lib.launch_count() - n0)

            def call(i, attn=attn, xs=xs, text=text, img=img, ac=ac):
                with _autocast(ac):
                    attn(xs[i], encoder_hidden_states=(text, img))
            arms[name] = {"call": call, "y": y, "launches": launches, "times": [], "keep": (attn, proc, xs, text, img)}
        xc = arms["ac_f32_x"]["keep"][2]
        conv = {"call": lambda i: ops.convert(xc[i], BF16), "times": []}
        for _ in range(rounds):
            for name in ARMS:
                with torch.no_grad():
                    arms[name]["times"].append(bench._graph_time_us(arms[name]["call"], nbuf))
            conv["times"].append(bench._graph_time_us(conv["call"], nbuf))
        row = {}
        for name in ARMS:
            row[f"{name}_us"] = round(statistics.median(arms[name]["times"]), 2)
            row[f"{name}_us_all"] = [round(t, 2) for t in arms[name]["times"]]
            row[f"{name}_launches_per_call"] = arms[name]["launches"]
        row["convert_x_us"] = round(statistics.median(conv["times"]), 2)
        row["convert_x_bytes"] = x32.numel() * 6
        ref = arms["bf16"]["y"]
        for name in ("ac_bf16_x", "ac_f32_x"):
            row[f"{name}_equals_bf16"] = bool(torch.equal(arms[name]["y"], ref))
        row["max_abs_f32_vs_bf16"] = float((arms["f32"]["y"].float() - ref.float()).abs().max())
        shapes[f"S{S}_C{C}"] = row
        print(f"S={S:5d} C={C:5d}  " + "  ".join(f"{n} {row[n + '_us']:8.2f}" for n in ARMS)
              + f"  convert_x {row['convert_x_us']:.2f} us  launches " + "/".join(str(row[n + '_launches_per_call']) for n in ARMS),
              flush=True)
        for arm in arms.values():
            arm["keep"][1].enable_kv_cache(False)
        del arms, conv, xc
        torch.cuda.empty_cache()
    return shapes


def train_step_ms(dev, batch, steps, warmup):
    import photoverse_b200 as pv
    from photoverse_b200.host.text_encoder import ConceptTextEncoder
    from photoverse_b200.host.train_step import Trainer, synthetic_train_batch
    from photoverse_b200.host.unet_sd15 import UNetSD15
    from photoverse_b200.lora import inject_lora
    torch.backends.cudnn.benchmark = True
    out = {}
    for name in ("bench_bf16_backbone", "f32_unet_bf16_autocast"):
        torch.manual_seed(0)
        unet = UNetSD15()
        pv.set_visual_cross_attention_adapter(unet, num_tokens=(5,))
        ia, ta = pv.PhotoVerseAdapter(num_tokens=5), pv.PhotoVerseAdapter(num_tokens=5)
        te = ConceptTextEncoder()
        unet.requires_grad_(False)
        te.requires_grad_(False)
        inject_lora(unet, r=8, lora_dropout=0.0)
        if name == "bench_bf16_backbone":          # bench.py --workload train
            unet.to(device=dev, dtype=BF16).to(memory_format=torch.channels_last)
            te.to(device=dev, dtype=BF16).eval()
            for n, p in unet.named_parameters():
                if "to_k_ip" in n or "to_v_ip" in n or "lora_" in n:
                    p.data = p.data.float()
            data_dt, ac = BF16, None
        else:
            unet.to(device=dev).to(memory_format=torch.channels_last)
            te.to(device=dev).eval()
            data_dt, ac = F32, BF16
        for n, p in unet.named_parameters():
            if "to_k_ip" in n or "to_v_ip" in n or "lora_" in n:
                p.requires_grad_(True)
        for m in (ia, ta):
            m.to(dev)
        unet.eval()
        tr = Trainer(unet, ia, ta, text_encoder=te, autocast_dtype=ac)
        b = synthetic_train_batch(batch, 64, seed=100, device=dev, dtype=data_dt)
        torch.manual_seed(1000)
        try:
            for _ in range(warmup):
                tr.step(b)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                loss, _ = tr.step(b)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3 / steps
            out[name] = {"ms_per_step": round(ms, 2), "final_loss": round(float(loss), 5), "batch": batch, "steps": steps}
        except Exception as e:                      # recorded, not hidden: the other arm still runs
            out[name] = {"error": f"{type(e).__name__}: {e}"[:400]}
        print(name, out[name], flush=True)
        del tr, unet, ia, ta, te, b
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=16)
    ap.add_argument("--li", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--train-batch", type=int, default=16)
    ap.add_argument("--train-steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("autocast_bench.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    res = {"device": torch.cuda.get_device_name(dev), "rows": a.rows, "li": a.li, "lt": bench.LT}
    res["convert"] = convert_bandwidth(dev)
    res["shapes"] = layer_times(dev, a.rows, a.li, a.rounds)
    tot = {n: sum(res["shapes"][f"S{S}_C{C}"][f"{n}_us"] for S, C in bench.LAYER_SHAPES) for n in ARMS + ("convert_x",)}
    res["unet_eval_16_layers_us"] = {n: round(t, 1) for n, t in tot.items()}
    res["unet_eval_convert_x_bytes"] = sum(res["shapes"][f"S{S}_C{C}"]["convert_x_bytes"] for S, C in bench.LAYER_SHAPES)
    print(json.dumps(res["unet_eval_16_layers_us"]), flush=True)
    res["train_step"] = train_step_ms(dev, a.train_batch, a.train_steps, 3)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
