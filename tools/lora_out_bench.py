"""What a LoRA on the cross-attention out projection (``attn2.to_out.0``) costs, next to the q/k/v-only LoRA of the
reference recipe.

  * training step (ms) of bench.py's training configuration (full SD-1.5 UNet, bf16 backbone, float32 masters of the
    trainable set, CLIP text tower with concept injection, batch `--train-batch`, latent 64^2, LoRA dropout 0), LoRA on
    q/k/v against LoRA on q/k/v/out, at r = 8 and r = 128; the two arms of a rank alternate `--rounds` times, each round
    timing `--steps` steps with CUDA events after `--warmup` steps; median per arm.  With an out-projection LoRA each
    layer re-packs and re-transposes Wo every step and adds one pv_lora_bwd (r <= 16) or the GEMM route (r = 128);
  * generation images/s of the CUDA-graph GenerationEngine (batch `--gen-batch`, latent 64^2, `--gen-steps` DDIM steps),
    a merged LoRA (r = 8) on q/k/v against one on q/k/v/out, alternating `--rounds` times; kernels per UNet evaluation.
Usage: python tools/lora_out_bench.py [--train-batch 16] [--rounds 3] [--steps 10] [--out FILE.json]"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

BF16 = torch.bfloat16
ARMS = {"qkv": ("attn2.to_k", "attn2.to_v", "attn2.to_q"),
        "qkv_out": ("attn2.to_k", "attn2.to_v", "attn2.to_q", "attn2.to_out.0")}


def _trainer(dev, targets, r, batch):
    import photoverse_b200 as pv
    from photoverse_b200.host.text_encoder import ConceptTextEncoder
    from photoverse_b200.host.train_step import Trainer, synthetic_train_batch
    from photoverse_b200.host.unet_sd15 import UNetSD15
    from photoverse_b200.lora import inject_lora
    torch.manual_seed(0)
    unet = UNetSD15()
    pv.set_visual_cross_attention_adapter(unet, num_tokens=(5,))
    ia, ta = pv.PhotoVerseAdapter(num_tokens=5), pv.PhotoVerseAdapter(num_tokens=5)
    te = ConceptTextEncoder()
    unet.requires_grad_(False)
    te.requires_grad_(False)
    inject_lora(unet, r=r, target_modules=targets)
    unet.to(device=dev, dtype=BF16).to(memory_format=torch.channels_last)
    te.to(device=dev, dtype=BF16).eval()
    for m in (ia, ta):
        m.to(dev)
    for n, p in unet.named_parameters():
        if "to_k_ip" in n or "to_v_ip" in n or "lora_" in n:
            p.data = p.data.float()
            p.requires_grad_(True)
    unet.eval()
    tr = Trainer(unet, ia, ta, text_encoder=te)
    return tr, synthetic_train_batch(batch, 64, seed=100, device=dev, dtype=BF16)


def _time_steps(tr, b, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, _ = tr.step(b)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, float(loss)


def train_times(dev, batch, rounds, steps, warmup):
    out = {}
    for r in (8, 128):
        arms = {name: _trainer(dev, targets, r, batch) for name, targets in ARMS.items()}
        torch.manual_seed(1000)
        for tr, b in arms.values():
            for _ in range(warmup):
                tr.step(b)
        torch.cuda.synchronize()
        times = {name: [] for name in arms}
        loss = {}
        for _ in range(rounds):
            for name, (tr, b) in arms.items():
                ms, loss[name] = _time_steps(tr, b, steps)
                times[name].append(round(ms, 3))
        row = {f"{name}_ms_per_step": round(statistics.median(t), 3) for name, t in times.items()}
        row.update({f"{name}_ms_all": t for name, t in times.items()})
        row.update({f"{name}_final_loss": round(v, 5) for name, v in loss.items()})
        row["extra_ms_per_step"] = round(row["qkv_out_ms_per_step"] - row["qkv_ms_per_step"], 3)
        row["trainable_elements"] = {name: arms[name][0].buf.numel() for name in arms}
        out[f"lora_r{r}"] = row
        print(f"train r={r}: " + json.dumps(row), flush=True)
        del arms
        torch.cuda.empty_cache()
    return out


def gen_rates(dev, batch, gen_steps, rounds):
    import photoverse_b200 as pv
    from photoverse_b200.host.pipeline import GenerationEngine, synthetic_inputs
    from photoverse_b200.host.unet_sd15 import UNetSD15
    from photoverse_b200.lora import inject_lora
    engines = {}
    for name, targets in ARMS.items():
        torch.manual_seed(0)
        unet = UNetSD15()
        pv.set_visual_cross_attention_adapter(unet, num_tokens=(5,))
        ia, ta = pv.PhotoVerseAdapter(num_tokens=5), pv.PhotoVerseAdapter(num_tokens=5)
        inject_lora(unet, r=8, target_modules=targets)
        g = torch.Generator().manual_seed(1)
        with torch.no_grad():
            for n, p in unet.named_parameters():
                if "lora_B" in n:
                    p.copy_(0.05 * torch.randn(p.shape, generator=g))
        for m in (unet, ia, ta):
            m.requires_grad_(False).eval().to(device=dev, dtype=BF16)
        unet.to(memory_format=torch.channels_last)
        eng = GenerationEngine(unet, ia, ta, batch=batch, latent=64, num_steps=gen_steps, dtype=BF16, device=dev)
        eng.load_inputs(synthetic_inputs(batch, 64, seed=5, device=dev, dtype=BF16))
        eng.generate()
        torch.cuda.synchronize()
        engines[name] = eng
    times = {name: [] for name in engines}
    for _ in range(rounds):
        for name, eng in engines.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            eng.generate()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(round(batch / (e0.elapsed_time(e1) * 1e-3), 4))
    row = {f"{name}_images_per_s": statistics.median(t) for name, t in times.items()}
    row.update({f"{name}_images_per_s_all": t for name, t in times.items()})
    row.update({f"{name}_launches_per_unet_eval": eng.launches_per_eval for name, eng in engines.items()})
    row.update({"batch": batch, "denoise_steps": gen_steps})
    print("generate: " + json.dumps(row), flush=True)
    for eng in engines.values():
        eng.close()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--train-batch", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--gen-batch", type=int, default=8)
    ap.add_argument("--gen-steps", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lora_out_bench.py measures on the GPU; no CUDA device found")
    dev = torch.device("cuda:0")
    torch.backends.cudnn.benchmark = True
    res = {"device": torch.cuda.get_device_name(dev), "train_batch": a.train_batch, "rounds": a.rounds,
           "steps_per_round": a.steps}
    res["train_step"] = train_times(dev, a.train_batch, a.rounds, a.steps, a.warmup)
    res["generate"] = gen_rates(dev, a.gen_batch, a.gen_steps, a.rounds)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
