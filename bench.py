#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config, on N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

--dump-outputs DIR is available for the generate workload of --impl ours only; with --workload train or
--impl reference it is rejected.

Workload (config 2 of BASELINE.json): 50-step DDIM generation at 512^2 (latent 64^2), batch 8 per GPU, bf16,
guidance 1.0, SD-1.5-shaped UNet + PhotoVerse adapters, random-init weights, synthetic encoder outputs.
One bench "step" = ONE full generation of the per-GPU batch: image/text adapters once, K/V projection of the 16
attn2 layers once, then 50 denoising steps, each evaluating the UNet on the unconditional AND the conditional
branch as the reference does (models/infer.py:103-114) -- here as one doubled-batch call.

Reported on one JSON line (rank 0):
  value      images/s, inputs already resident in HBM, CUDA-event timed, max over ranks
  e2e        same metric through the public API with HOST (pinned) inputs: H2D of every input + D2H of the latents
             inside the timed region
  roofline   the fused Q-projection + dual-branch attention kernel (the dominant native kernel), timed alone with
             CUDA events over the 16 attn2 layer shapes of one UNet evaluation, against the measured bf16 peak; next to
             it the whole processor call (one launch / two launches) and the SAME-BOX GPU-EAGER comparator: the
             reference's own op sequence (attention_processor.py:297-433: cuBLASLt linears + two SDPA calls) in bf16
  train      BASELINE config[3] as a sub-record at every N (ms/step, samples/s, exposed allreduce time) for LoRA rank
             8 and 128, so that the driver's 1 -> 8 GPU runs carry the NCCL-limited training curve too
  cfg3       (N >= 2) BASELINE config[2]: guidance 7.5, global batch 64 strong-scaled over the N GPUs
  cpu_baseline  the oracle port of the reference path, host UNet in fp32 on the host cores, bounded sample
  --impl reference : the CPU arm as the whole job (same metric / config keys), rank 0 only.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

# stdout carries exactly ONE JSON line: NCCL's own messages (e.g. the "NCCL version ..." banner that NCCL_DEBUG=VERSION
# prints on the first communicator) go to stderr.
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec @50 steps 512^2; dual-branch cross-attn TFLOP/s as % of B200 peak"
LAYER_SHAPES = [(4096, 320)] * 5 + [(1024, 640)] * 5 + [(256, 1280)] * 5 + [(64, 1280)]   # (S, C) of the 16 attn2 layers
LT = 77


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="images per GPU per generation")
    ap.add_argument("--denoise-steps", type=int, default=50)
    ap.add_argument("--latent", type=int, default=64)
    ap.add_argument("--token-index", default="0", help="adapter head used at inference (reference default 0) or 'full'")
    ap.add_argument("--mode", default="batched", choices=["batched", "two_call", "cond_only"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train-leg", action="store_true", help="skip the config[3] training sub-records")
    ap.add_argument("--no-cfg3-leg", action="store_true", help="skip the config[2] CFG 7.5 strong-scaling sub-record")
    ap.add_argument("--train-steps", type=int, default=20, help="timed steps of each training sub-record")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--nchw", action="store_true", help="keep the host UNet in NCHW (default: channels_last)")
    ap.add_argument("--stock-epilogues", action="store_true",
                    help="stock PyTorch GroupNorm / SiLU / GEGLU in the host UNet instead of the pv_backbone.cu kernels (A/B)")
    ap.add_argument("--workload", default="generate", choices=["generate", "train"],
                    help="generate: BASELINE config[1] (the headline line);  train: config[3] training step")
    ap.add_argument("--train-batch", type=int, default=16, help="samples per GPU per training step (config[3])")
    ap.add_argument("--lora-rank", type=int, default=8)
    ap.add_argument("--lora-dropout", type=float, default=0.0,
                    help="train workload: peft lora_dropout (reference default 0.1; 0 = SURVEY config 4 parity setting)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="generate workload: write the latents of the last timed generation (rank 0) to DIR/latents.npy "
                         "in float32, so that two builds can be compared output for output on the same seeded inputs "
                         "(with a tolerance: two runs of one build are not bit-identical, see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "generate" or args.impl != "ours"):
        ap.error("--dump-outputs applies to the generate workload of --impl ours")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """DIR/<name>.npy in float32.  An array larger than what is left of DUMP_LIMIT_BYTES keeps its leading samples
    (first dimension) only, so a dump stays comparable between runs of the same arguments.
    Two processes of one build on one B200 (1000 W power limit; default batch 8, latent 64, 50 steps; --steps / --warmup
    3 / 2 against 2 / 1) gave latents of rms 13.6 that agreed exactly in 73 % of the elements, with an rms difference
    of 0.07 and a largest difference of 2.25; compare dumps with a tolerance, not bitwise."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_LIMIT_BYTES
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        rows = min(a.shape[0], left // max(1, a[:1].nbytes))
        np.save(os.path.join(out_dir, name + ".npy"), a[:rows])
        left -= a[:rows].nbytes


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"bf16_tflops": float(d["bf16_tflops"]), "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "hbm_gbs": float(d["hbm_gbs"]), "source": "measured"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [x for x in sm if x >= 0.5 * max(sm)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------
# model construction (identical seeds on both arms)
# ------------------------------------------------------------------------------------------------------------
def build_models(device, dtype, T=5, channels_last=True):
    import photoverse_b200 as pv
    torch.backends.cudnn.benchmark = True
    from photoverse_b200.host.unet_sd15 import UNetSD15
    torch.manual_seed(0)
    unet = UNetSD15()
    pv.set_visual_cross_attention_adapter(unet, num_tokens=(T,))
    image_adapter = pv.PhotoVerseAdapter(num_tokens=T)
    text_adapter = pv.PhotoVerseAdapter(num_tokens=T)
    for m in (unet, image_adapter, text_adapter):
        m.requires_grad_(False)
        m.eval()
        m.to(device=device, dtype=dtype)
    if channels_last:      # host-model plumbing: NHWC activations for the cuDNN convolutions of the backbone
        unet.to(memory_format=torch.channels_last)
    return unet, image_adapter, text_adapter


# ------------------------------------------------------------------------------------------------------------
# roofline leg: the fused attention kernel alone, per attn2 layer shape, CUDA-event timed
# ------------------------------------------------------------------------------------------------------------
def attn_kernel_flops(rows_b, S, C, Li):
    return 2 * rows_b * S * C * C + 4 * rows_b * S * C * (LT + Li)      # Q projection + QK^T + PV (SURVEY 8d terms)


def processor_flops_cached(rows_b, S, C, Li):
    return 4 * rows_b * S * C * C + 4 * rows_b * S * C * (LT + Li)      # + out projection; K/V cached across steps


def eager_reference_processor(x, text, img, wq, wk, wv, wkip, wvip, wo, bo, H):
    """The reference's no-grad call, op for op, in PyTorch eager (the kernels to beat on this box, SURVEY 2.2 P1-P15):
    attention_processor.py:297 to_q, :304-305 to_k / to_v, :310-313 split heads, :317-319 SDPA(text), :321-322 merge,
    :392-396 to_k_ip / to_v_ip, :397 norm side output, :400-407 SDPA(image), :412 add, :423 to_out, :433 rescale.
    K/V are projected on every call, as the reference does (SURVEY D7)."""
    import torch.nn.functional as F
    B, _, C = x.shape
    d = C // H
    heads = lambda t: t.view(B, -1, H, d).transpose(1, 2)
    q = heads(F.linear(x, wq))
    k, v = heads(F.linear(text, wk)), heads(F.linear(text, wv))
    o = F.scaled_dot_product_attention(q, k, v, attn_mask=None, dropout_p=0.0, is_causal=False)
    o = o.transpose(1, 2).reshape(B, -1, C).to(q.dtype)
    ik, iv = heads(F.linear(img, wkip)), heads(F.linear(img, wvip))
    vnorm = torch.norm(iv, dim=-1, keepdim=True)
    io = F.scaled_dot_product_attention(q, ik, iv, attn_mask=None, dropout_p=0.0, is_causal=False)
    io = io.transpose(1, 2).reshape(B, -1, C).to(q.dtype)
    o = o + io
    y = F.linear(o, wo, bo)
    return y / 1.0, vnorm


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant (S4096, C320) attention instance, read
    from the committed `ncu --set full` summary of this round (profiles/r02_ncu_attn.csv), else the round-1 one."""
    import csv
    for name in ("r02_ncu_attn.csv", "r01n_ncu_attn.csv"):
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        try:
            rows = list(csv.reader(open(path)))
            head, units = rows[0], rows[1]
            ir, iw, ik = head.index("dram__bytes_read.sum"), head.index("dram__bytes_write.sum"), head.index("Kernel Name")
            mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            for r in rows[2:]:
                if "<40" in r[ik]:          # head_dim 40 instance = the S4096 C320 layer
                    return (float(r[ir]) * mult[units[ir]] + float(r[iw]) * mult[units[iw]],
                            f"profiles/{name}: dram__bytes_read.sum + dram__bytes_write.sum, one launch of {r[ik][:60]}")
        except Exception:
            continue
    return None, "no committed ncu --set full summary"


def _graph_time_us(fn, nbuf, reps=20):
    """Device time per call: `reps` launches captured in a CUDA graph (as the generation engine runs them), so that the
    Python / ctypes launch rate does not bound kernels shorter than it; CUDA events around one replay."""
    for i in range(3):
        fn(i % nbuf)
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for i in range(reps):
            fn(i % nbuf)
    gr.replay()
    times = []
    for _ in range(3):                     # median of three replays: one replay is ~0.5 ms, short against a power-cap dip
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        gr.replay()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e3 / reps)
    return sorted(times)[1]


def roofline_leg(device, rows_b, Li, scale):
    """Returns roofline dict for the fused attention kernel + per-family detail + whole-processor numbers."""
    from photoverse_b200 import _lib, ops
    peaks = measured_peaks()
    dt = torch.bfloat16
    g = torch.Generator().manual_seed(1)
    fam = {}
    l2_bytes = 192 << 20
    lib = _lib.lib()
    for (S, C) in sorted(set(LAYER_SHAPES), reverse=True):
        H = 8
        text = torch.randn(rows_b, LT, 768, generator=g).to(device, dt)
        img = torch.randn(rows_b, Li, 768, generator=g).to(device, dt)
        wq = (torch.randn(C, C, generator=g) / C ** 0.5).to(device, dt)
        wo = (torch.randn(C, C, generator=g) / C ** 0.5).to(device, dt)
        bo = torch.zeros(C, device=device)
        wkv_t = (torch.randn(2 * C, 768, generator=g) / 768 ** 0.5).to(device, dt)
        wkv_i = (torch.randn(2 * C, 768, generator=g) / 768 ** 0.5).to(device, dt)
        kv = ops.kv_pack(text, img, wkv_t, wkv_i, H)
        xbytes = rows_b * S * C * 2
        nbuf = max(2, min(16, l2_bytes // max(1, 3 * xbytes) + 1))     # rotate X/O/Y sets larger than L2 in total
        xs = [torch.randn(rows_b, S, C, device=device, dtype=dt) for _ in range(nbuf)]
        os_ = [torch.empty_like(xs[0]) for _ in range(nbuf)]
        ys = [torch.empty_like(xs[0]) for _ in range(nbuf)]
        sync = torch.zeros(int(lib.pv_dual_attn_sync_words(rows_b, S)), device=device, dtype=torch.int32)

        def attn_only(i):
            _lib.check(lib.pv_dual_attn_core_fwd(1, ops._ptr(xs[i]), ops._ptr(wq), ops._ptr(kv.Kp), ops._ptr(kv.Vp),
                                                 ops._ptr(os_[i]), None, rows_b, S, C, H, LT, Li, 1.0, 1.0, ops._stream()))

        def full(i):
            _lib.check(lib.pv_dual_attn_fwd(1, ops._ptr(xs[i]), ops._ptr(wq), ops._ptr(kv.Kp), ops._ptr(kv.Vp),
                                            ops._ptr(wo), ops._ptr(bo), ops._ptr(ys[i]), None, ops._ptr(os_[i]), None,
                                            ops._ptr(sync), rows_b, S, C, H, LT, Li, 1.0, 1.0, ops._stream()))

        bo_b = bo.to(dt)
        eager_out = [None]

        def eager(i):        # the reference's op sequence; K/V recomputed per call like the reference (D7)
            eager_out[0] = eager_reference_processor(xs[i], text, img, wq, wkv_t[:C], wkv_t[C:], wkv_i[:C], wkv_i[C:], wo, bo_b, H)

        out = {"attn_us": _graph_time_us(attn_only, nbuf)}
        n0 = _lib.launch_count()
        full(0)
        out["launches_per_call"] = int(_lib.launch_count() - n0)
        out["proc_us"] = _graph_time_us(full, nbuf)                     # the library's default policy
        for opt, key in ((2, "proc_one_launch_us"), (0, "proc_two_launch_us")):
            if S > 128:
                _lib.set_option("fuse_out", opt)
                out[key] = _graph_time_us(full, nbuf)
        _lib.set_option("fuse_out", 1)
        with torch.no_grad():
            out["gpu_eager_us"] = _graph_time_us(eager, nbuf)
            full(0)
            eager(0)
            out["eager_vs_ours_max_abs"] = float((eager_out[0][0].float() - ys[0].float()).abs().max())
        out["speedup_vs_gpu_eager"] = out["gpu_eager_us"] / out["proc_us"]
        fam[f"S{S}_C{C}"] = out
        del xs, os_, ys
    # attn1 (SURVEY 8 row f4): the opt-in self-attention kernel beside the stock SDPA call it would replace, same inputs
    attn1 = {}
    for (S, C) in sorted(set(LAYER_SHAPES), reverse=True):
        H = 8
        qkv = torch.randn(rows_b, S, 3 * C, generator=g).to(device, dt)
        q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
        hd = lambda t: t.reshape(rows_b, S, H, C // H).transpose(1, 2)
        with torch.no_grad():
            t_ours = _graph_time_us(lambda i: ops.self_attn(q, k, v, H), 1, reps=10)
            t_sdpa = _graph_time_us(lambda i: torch.nn.functional.scaled_dot_product_attention(hd(q), hd(k), hd(v)), 1, reps=10)
        attn1[f"S{S}_C{C}"] = {"ours_us": round(t_ours, 1), "sdpa_us": round(t_sdpa, 1), "ratio": round(t_sdpa / t_ours, 2)}
        del qkv
    # aggregate over the 16 layers of one UNet evaluation
    tsum = lambda key: sum(fam[f"S{S}_C{C}"][key] for S, C in LAYER_SHAPES) * 1e-6
    t_attn, t_proc, t_eager = tsum("attn_us"), tsum("proc_us"), tsum("gpu_eager_us")
    f_attn = sum(attn_kernel_flops(rows_b, S, C, Li) for S, C in LAYER_SHAPES)
    f_proc = sum(processor_flops_cached(rows_b, S, C, Li) for S, C in LAYER_SHAPES)
    ach = f_attn / t_attn / 1e12
    traffic, traffic_src = ncu_traffic()
    roof = {"bound": "tensor", "kernel": "dual_attn_fwd_pair_roles_kernel (head_dim 40 / 80 layers) / dual_attn_fwd_pair_kernel (head_dim 160): fused Q-proj + dual-branch attention on cta_group::2 CTA pairs (attention phase only: pv_dual_attn_core_fwd); single-CTA persistent kernel for S <= 128",
            "achieved": round(ach, 2), "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
            "frac": round(ach / peaks["bf16_tflops"], 4), "peak_source": peaks["source"] + " cuBLAS bf16 burst",
            "traffic": traffic, "traffic_unit": "bytes per launch, S4096_C320 layer", "traffic_source": traffic_src,
            "how": f"CUDA events around a CUDA graph of 20 launches per attn2 layer shape at {rows_b} rows (uncond+cond), median of 3 replays, "
                   f"inputs rotated through > L2 of buffers; aggregated over the 16 layers of one UNet evaluation; "
                   f"algorithmic FLOPs = 2 rows C^2 + 4 rows C (77 + Li) per launch (processor: 4 rows C^2 + ...); "
                   f"proc_us = whole processor call with the library's default launch policy (one launch for C <= 320, "
                   f"attention + out-projection launches otherwise), proc_one/two_launch_us = both forms forced; "
                   f"gpu_eager_us = the reference's own op sequence in PyTorch eager bf16 on this GPU (cuBLASLt + 2 SDPA, "
                   f"K/V projected per call), graph-replayed like ours",
            "per_shape_us": {k: {kk: (round(vv, 2) if isinstance(vv, float) else vv) for kk, vv in v.items()} for k, v in fam.items()},
            "processor_tflops": round(f_proc / t_proc / 1e12, 2),
            "processor_frac": round(f_proc / t_proc / 1e12 / peaks["bf16_tflops"], 4),
            "processor_ms_per_unet_eval": round(t_proc * 1e3, 3),
            "gpu_eager_ms_per_unet_eval": round(t_eager * 1e3, 3),
            "speedup_vs_gpu_eager": round(t_eager / t_proc, 2),
            "attn1_self_attention": {"note": "pv_self_attn_fwd (opt-in SelfAttnProcessor, NOT used by the benchmarked step) vs the stock "
                                             "F.scaled_dot_product_attention it would replace; ratio > 1 = ours faster",
                                     "per_shape": attn1}}
    return roof


# ------------------------------------------------------------------------------------------------------------
# CPU arm: oracle port of the reference path on the host cores
# ------------------------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, denoise_steps, latent, token_index, batch, T=5):
    """Each step = bounded sample of the SAME workload: the whole batch, adapters once + ONE of the `denoise_steps`
    denoise steps (uncond + cond UNet evaluation as two calls, like infer.py:103-114), fp32 on all host cores."""
    from oracle.host_reference import clone_adapter_as_oracle, clone_with_oracle_processors
    from photoverse_b200.host.ddim import make_ddim_schedule
    from photoverse_b200.host.pipeline import synthetic_inputs
    import photoverse_b200 as pv
    from photoverse_b200.host.unet_sd15 import UNetSD15
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    unet = UNetSD15()
    pv.set_visual_cross_attention_adapter(unet, num_tokens=(T,))
    unet = clone_with_oracle_processors(unet).eval()
    torch.manual_seed(1)
    image_adapter = clone_adapter_as_oracle(pv.PhotoVerseAdapter(num_tokens=T)).eval()
    text_adapter = clone_adapter_as_oracle(pv.PhotoVerseAdapter(num_tokens=T)).eval()
    inp = synthetic_inputs(batch, latent, seed=0, dtype=torch.float32)
    sched = make_ddim_schedule(denoise_steps)
    t_ad, t_step = [], []
    with torch.no_grad():
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            text_adapter(inp.clip_hidden, token_index=token_index)
            img = image_adapter(inp.clip_hidden, token_index=token_index)
            img_u = image_adapter(inp.clip_hidden_uncond, token_index=token_index)
            t1 = time.perf_counter()
            lat = inp.noise
            t = torch.tensor([float(sched.timesteps[0])])
            eu = unet(lat, t, encoder_hidden_states=(inp.text_uncond, img_u)).sample     # infer.py:103-107
            ec = unet(lat, t, encoder_hidden_states=(inp.text, img)).sample              # infer.py:110-114
            eps = eu + 1.0 * (ec - eu)
            lat = sched.c_x[0] * lat + sched.c_eps[0] * eps
            t2 = time.perf_counter()
            if it >= warmup:
                t_ad.append(t1 - t0)
                t_step.append(t2 - t1)
    ad, st = statistics.mean(t_ad), statistics.mean(t_step)
    per_batch_s = ad + denoise_steps * st
    return {"images_per_s": batch / per_batch_s, "cores": cores, "adapter_s": ad, "denoise_step_s": st, "batch": batch,
            "sample": f"batch {batch} (the benchmarked batch): adapters once + 1 of {denoise_steps} DDIM steps (uncond + cond "
                      f"UNet evaluations), fp32, {cores} threads; generation time taken as adapters + {denoise_steps} x step; "
                      f"mean of {steps} after {warmup} warm-up"}


def train_leg(args, rank, world, device, lora_rank, steps, warmup, lora_dropout=0.0):
    """BASELINE config[3]: one training step = text / image adapters (5 heads) -> CLIP text tower with the concept
    embeddings injected (train.py:495-499) -> UNet forward in grad mode (16 processors, stochastic fusion) -> backward
    into the trainable set {adapters, to_k_ip / to_v_ip, LoRA A/B}, bucketed NCCL allreduce launched under the backward
    pass, per-group clipping, AdamW.  bf16 backbone, fp32 masters for the trainable set.  Weak scaling: batch per GPU
    fixed.  Returns the sub-record (rank 0) -- timing = CUDA events, max over ranks."""
    import torch.distributed as dist
    import photoverse_b200 as pv
    from photoverse_b200 import _lib
    from photoverse_b200.host.text_encoder import ConceptTextEncoder
    from photoverse_b200.host.train_step import Trainer, synthetic_train_batch
    from photoverse_b200.host.unet_sd15 import UNetSD15
    from photoverse_b200.lora import inject_lora
    torch.backends.cudnn.benchmark = True
    torch.manual_seed(0)
    unet = UNetSD15()
    pv.set_visual_cross_attention_adapter(unet, num_tokens=(5,))
    ia, ta = pv.PhotoVerseAdapter(num_tokens=5), pv.PhotoVerseAdapter(num_tokens=5)
    te = ConceptTextEncoder()
    unet.requires_grad_(False)
    te.requires_grad_(False)
    inject_lora(unet, r=lora_rank, lora_dropout=lora_dropout)
    unet.to(device=device, dtype=torch.bfloat16).to(memory_format=torch.channels_last)
    te.to(device=device, dtype=torch.bfloat16).eval()
    for m in (ia, ta):
        m.to(device)
    for n, p in unet.named_parameters():
        if "to_k_ip" in n or "to_v_ip" in n or "lora_" in n:
            p.data = p.data.float()                       # fp32 masters for the trainable set
            p.requires_grad_(True)
    unet.eval()
    if args.stock_epilogues:
        unet.set_fused_epilogues(False)                       # A/B: stock GroupNorm / SiLU in the frozen backbone
    if lora_dropout > 0:
        pv.unet.set_cross_attention_layers_to_train(unet)     # train.py:462 (activates the LoRA dropout)
    tr = Trainer(unet, ia, ta, text_encoder=te)
    b = synthetic_train_batch(args.train_batch, args.latent, seed=100 + rank, device=device, dtype=torch.bfloat16)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    torch.manual_seed(1000 + rank)
    for _ in range(warmup):
        tr.step(b)
    barrier()
    sampler = ClockSampler(device.index or 0)
    sampler.start()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ar = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    overlapped = 0
    e0.record()
    for k in range(steps):
        tr.reducer_events = ar[k]          # Trainer.step brackets reducer.finish() (the exposed part of the allreduce)
        loss, _ = tr.step(b)
        overlapped += tr.buckets_overlapped
    e1.record()
    barrier()
    clocks = sampler.stop()
    exposed = sum(a.elapsed_time(b_) for a, b_ in ar) / steps
    t = torch.tensor([e0.elapsed_time(e1), exposed], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, exposed = t.tolist()
    rec = {"metric": "training samples/s, adapter + LoRA + to_k_ip/to_v_ip step through dual-branch attention (config[3])",
           "value": round(args.train_batch * world * steps / (ms * 1e-3), 3), "unit": "samples/s", "n_gpus": world,
           "steps": steps, "warmup": warmup, "ms_per_step": round(ms / steps, 3), "scaling": "weak", "dtype": "bf16",
           "lora_rank": lora_rank, "lora_dropout": lora_dropout, "batch_per_gpu": args.train_batch, "latent": args.latent,
           "grad_elements": tr.buf.numel(), "allreduce": "bucketed slices of one flat fp32 buffer (+ touched flags), launched from "
           "autograd hooks under the backward pass; NCCL sum, / world",
           "allreduce_exposed_ms": round(exposed, 3), "buckets": len(tr.reducer.buckets),
           "buckets_launched_under_backward_per_step": round(overlapped / steps, 2),
           "text_encoder": "12-layer CLIP text tower with concept-token injection (train.py:495-499)",
           "gpu_launches": int(_lib.launch_count() - n0), "clocks": clocks, "final_loss": round(float(loss), 5)}
    del tr, unet, ia, ta, te, b
    torch.cuda.empty_cache()
    return rec


def run_train(args, rank, world, local_rank):
    """`--workload train`: config[3] as the whole job (one JSON line)."""
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    rec = train_leg(args, rank, world, device, args.lora_rank, args.steps, args.warmup, args.lora_dropout)
    if rank == 0:
        rec.update({"higher_is_better": True, "vs_baseline": None, "data": "synthetic",
                    "config": {"workload": f"config[3]: training step, batch {args.train_batch}/GPU, latent {args.latent}^2, Li=5, "
                                           f"LoRA r={args.lora_rank} (dropout {args.lora_dropout}) on attn2.to_q/k/v, fwd+bwd through 16 "
                                           f"processors + 2 adapters + CLIP text tower, overlapped NCCL allreduce of "
                                           f"{rec['grad_elements']} fp32 gradients, per-group clip, AdamW",
                               "batch_per_gpu": args.train_batch, "grad_elements": rec["grad_elements"]}})
        print(json.dumps(rec), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def shard_inputs(global_batch, world, rank, latent, dtype):
    """Pinned host inputs of this rank's shard; every sample is drawn from its GLOBAL index (sample_seeds), so the
    generated latents do not depend on the number of ranks."""
    from photoverse_b200.host.parallel import sample_seeds
    from photoverse_b200.host.pipeline import GenInputs, synthetic_inputs
    parts = [synthetic_inputs(1, latent, seed=sd, dtype=dtype) for sd in sample_seeds(100, global_batch, world, rank)]
    cat = lambda ts: torch.cat(ts).contiguous().pin_memory()
    T = len(parts[0].clip_hidden)
    return GenInputs([cat([p.clip_hidden[k] for p in parts]) for k in range(T)],
                     [cat([p.clip_hidden_uncond[k] for p in parts]) for k in range(T)],
                     cat([p.text for p in parts]), cat([p.text_uncond for p in parts]), cat([p.noise for p in parts]))


def cfg3_leg(args, rank, world, device, models, token_index):
    """BASELINE config[2]: classifier-free guidance 7.5, GLOBAL batch 64 (128 UNet rows per step) sharded over the N
    GPUs -- strong scaling, no collective in the loop.  One warm-up + one timed generation."""
    import torch.distributed as dist
    from photoverse_b200.host.pipeline import GenerationEngine
    from photoverse_b200.host.parallel import shard_range
    gb = 64
    b0, b1 = shard_range(gb, world, rank)
    unet, image_adapter, text_adapter = models
    eng = GenerationEngine(unet, image_adapter, text_adapter, b1 - b0, args.latent, args.denoise_steps, 7.5, token_index,
                           "batched", torch.bfloat16, device)
    host = shard_inputs(gb, world, rank, args.latent, torch.bfloat16)
    eng.load_inputs(host)
    eng.generate()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    lat = eng.generate()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    finite = bool(torch.isfinite(lat.float()).all().item())
    eng.close()
    del eng
    torch.cuda.empty_cache()
    return {"workload": "config[2]: CFG guidance 7.5, global batch 64 (doubled to 128 UNet rows), 50-step DDIM, sharded "
                        f"{gb // world} per GPU", "value": round(gb / (ms * 1e-3), 4), "unit": "images/s", "scaling": "strong",
            "global_batch": gb, "n_gpus": world, "ms_per_generation": round(ms, 2), "timed_generations": 1, "finite_output": finite}


def main():
    args = parse()
    token_index = args.token_index if args.token_index == "full" else int(args.token_index)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    Li = 5 if token_index == "full" else 1
    config = {"workload": f"config[1]: {args.denoise_steps}-step DDIM generation, batch {args.batch}/GPU, latent "
                          f"{args.latent}^2 (512^2 px), guidance 1.0, SD-1.5-shaped UNet (random init) + PhotoVerse "
                          f"processors on 16 attn2 layers + image/text adapters",
              "batch_per_gpu": args.batch, "denoise_steps": args.denoise_steps, "latent": args.latent,
              "unet_evals_per_step": "uncond+cond (reference infer.py:103-114)", "image_tokens": Li,
              "token_index": token_index, "l2": "step working set >> L2 (126 MB); roofline leg rotates buffers > L2"}
    # how THIS arm runs the UNet's normalisation / activation / residual glue (the workload above is the same on every arm)
    backbone_epilogues = ("stock PyTorch ops" if (args.stock_epilogues or args.nchw or args.impl != "ours")
                          else "photoverse_b200 kernels (pv_backbone.cu): channels-last GroupNorm+SiLU, LayerNorm, GEGLU, bias / residual sums")

    if args.workload == "train" and args.impl == "ours":
        return run_train(args, rank, world, local_rank)
    if args.impl == "reference":
        if rank != 0:
            return 0
        r = cpu_reference_run(args.steps, args.warmup, args.denoise_steps, args.latent, token_index, args.batch)
        config["cpu_sample_batch"] = r["batch"]
        line = {"impl": "reference", "metric": METRIC, "value": round(r["images_per_s"], 6), "unit": "images/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round((r["adapter_s"] + r["denoise_step_s"]) * 1e3, 3), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": round(r["images_per_s"], 6), "unit": "images/s", "cores": r["cores"],
                                 "kind": "port", "sample": r["sample"]},
                "e2e": {"value": round(r["images_per_s"], 6), "unit": "images/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return 0

    import torch.distributed as dist
    from photoverse_b200 import _lib
    from photoverse_b200.host.pipeline import GenerationEngine
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: photoverse_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- CPU baseline (rank 0, N == 1 only) before the GPU section ----
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(1, 1, args.denoise_steps, args.latent, token_index, args.batch)
        cpu_base = {"value": round(r["images_per_s"], 6), "unit": "images/s", "cores": r["cores"], "kind": "port",
                    "sample": r["sample"], "denoise_step_s": round(r["denoise_step_s"], 3), "batch": r["batch"]}

    dtype = torch.bfloat16
    unet, image_adapter, text_adapter = build_models(device, dtype, channels_last=not args.nchw)
    if args.stock_epilogues:
        unet.set_fused_epilogues(False)
    eng = GenerationEngine(unet, image_adapter, text_adapter, args.batch, args.latent, args.denoise_steps, 1.0,
                           token_index, args.mode, dtype, device, use_cuda_graph=not args.no_graph)
    host = shard_inputs(args.batch * world, world, rank, args.latent, dtype)       # per-sample seeds by GLOBAL index
    h2d = host.nbytes()
    out_host = torch.empty(args.batch, 4, args.latent, args.latent, dtype=dtype).pin_memory()
    d2h = out_host.numel() * out_host.element_size()

    # ---- device-resident leg ("value") ----
    eng.load_inputs(host)
    for _ in range(args.warmup):
        lat = eng.generate()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    n0, r0 = _lib.launch_count(), eng.replays
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        lat = eng.generate()
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    launches = (_lib.launch_count() - n0) + (eng.replays - r0) * eng.launches_per_eval
    native_per_eval = eng.launches_per_eval
    finite = bool(torch.isfinite(lat.float()).all().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"latents": lat})

    # ---- end-to-end leg: host buffers in, host latents out, copies inside the timed region ----
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        eng.load_inputs(host)
        lat = eng.generate()
        out_host.copy_(lat, non_blocking=True)
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)

    t = torch.tensor([ms, ms_e2e], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()
    images = args.batch * world * args.steps
    value = images / (ms * 1e-3)
    e2e_value = images / (ms_e2e * 1e-3)

    roof = None
    if rank == 0:
        rows_b = 2 * args.batch if args.mode == "batched" else args.batch
        roof = roofline_leg(device, rows_b, Li, 1.0)
        # share of the generation spent in the native processor kernels (Amdahl note, SURVEY 8d)
        per_gen_proc_ms = roof["processor_ms_per_unet_eval"] * args.denoise_steps * (2 if args.mode == "two_call" else 1)
        roof["processor_share_of_step"] = round(per_gen_proc_ms / (ms / args.steps), 4)
    if world > 1:
        dist.barrier()
    # ---- sub-records: config[2] strong scaling (N >= 2) and config[3] training (every N) ----
    cfg3 = None
    if world > 1 and not args.no_cfg3_leg:
        cfg3 = cfg3_leg(args, rank, world, device, (unet, image_adapter, text_adapter), token_index)
    eng.close()
    del eng, unet, image_adapter, text_adapter
    torch.cuda.empty_cache()
    train = None
    if not args.no_train_leg:
        train = {f"lora_r{r}": train_leg(args, rank, world, device, r, args.train_steps, 3) for r in (8, 128)}
    if rank == 0:
        line = {"metric": METRIC, "value": round(value, 4), "unit": "images/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config,
                "roofline": roof, "cpu_baseline": cpu_base,
                "e2e": {"value": round(e2e_value, 4), "unit": "images/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h, "ms_per_step": round(ms_e2e / args.steps, 3)},
                "gpu_launches": int(launches), "clocks": clocks, "finite_output": finite,
                "native_kernels_per_unet_eval": native_per_eval, "backbone_epilogues": backbone_epilogues,
                "train": train, "cfg3": cfg3}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
