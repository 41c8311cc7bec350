"""GPU x2 (two B200s on one node): the data-parallel contracts of SURVEY 4.3 / 8e on real devices with NCCL --
  * generation: per-sample latents of a 2-rank run are BIT-IDENTICAL to one process generating the same two shards one
    after the other (samples are seeded by global index, shards are contiguous, there is no collective in the loop;
    invariance to the BATCH a sample is generated in is test_gpu_pipeline's engine test, to bf16 tolerance);
  * training: the allreduced gradients of a 2-rank step == the mean of the two single-rank gradients.
Skipped on a machine with fewer than two GPUs; the N > 1 host logic is covered on CPU by test_parallel_cpu."""
import json
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r"""
import json, os, sys
import torch, torch.distributed as dist
sys.path.insert(0, os.environ["PV_ROOT"])
import bench
from photoverse_b200.host.parallel import shard_range, trainable_named_parameters
from photoverse_b200.host.pipeline import GenerationEngine
from photoverse_b200.host.train_step import Trainer, synthetic_train_batch

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
out = {}
# ---- generation: global batch 4 sharded over the ranks ----
GB, LAT, STEPS = 4, 32, 6
unet, ia, ta = bench.build_models(dev, torch.bfloat16)
# separate processes must pick the same cuDNN / cuBLAS algorithms for the frozen backbone to be comparable bit for bit
torch.backends.cudnn.benchmark = False
torch.backends.cudnn.deterministic = True
out["latents"] = {}
eng = GenerationEngine(unet, ia, ta, GB // 2, LAT, STEPS, 3.0, 0, "batched", torch.bfloat16, dev)
for shard in ([0, 1] if world == 1 else [rank]):      # world 1: the two shards one after the other on one GPU
    b0, b1 = shard_range(GB, 2, shard)
    eng.load_inputs(bench.shard_inputs(GB, 2, shard, LAT, torch.bfloat16))
    lat = eng.generate().float().cpu()
    out["latents"].update({str(b0 + i): lat[i].flatten().tolist() for i in range(b1 - b0)})
eng.close()
del eng, unet, ia, ta
# ---- training: one step, gradients after the (overlapped) allreduce ----
import photoverse_b200 as pv
from photoverse_b200.host.unet_sd15 import UNetSD15
from photoverse_b200.lora import inject_lora
torch.manual_seed(0)
unet = UNetSD15(block_out_channels=(320, 640), layers_per_block=1)
pv.set_visual_cross_attention_adapter(unet, num_tokens=(5,))
ia, ta = pv.PhotoVerseAdapter(num_tokens=5), pv.PhotoVerseAdapter(num_tokens=5)
unet.requires_grad_(False)
inject_lora(unet, r=8)
g = torch.Generator().manual_seed(1)
for n, p in unet.named_parameters():
    if "to_k_ip" in n or "to_v_ip" in n:
        p.requires_grad_(True)
    if "lora_B" in n:
        with torch.no_grad():
            p.copy_(0.05 * torch.randn(p.shape, generator=g))
for m in (unet, ia, ta):
    m.to(dev)
unet.eval()
tr = Trainer(unet, ia, ta)
grads = {}
for shard in ([0, 1] if world == 1 else [rank]):              # world 1: both shards one after the other, no allreduce
    batch = synthetic_train_batch(2, latent=16, seed=40 + shard, device=dev, dtype=torch.float32)
    torch.manual_seed(70 + shard)                             # fusion-rule draws of that shard
    tr.opt.zero_grad(set_to_none=True)
    with torch.enable_grad():
        loss, _ = tr.loss(batch)
    tr.reducer.begin(tr.expected_gradients())
    loss.backward()
    tr.reducer.finish()
    tr.buf.unpack()
    grads[shard] = {n: (None if p.grad is None else p.grad.double().flatten()[:64].tolist()) for n, p in tr.named}
out["grads"] = grads
out["buckets_early"] = tr.buckets_overlapped
json.dump(out, open(os.path.join(os.environ["PV_OUT"], f"w{world}_r{rank}.json"), "w"))
dist.destroy_process_group()
"""


def _run(world, tmp):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = os.path.join(tmp, "worker.py")
    with open(script, "w") as f:
        f.write(WORKER)
    env = dict(os.environ, PV_ROOT=ROOT, PV_OUT=str(tmp))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), script]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return [json.load(open(os.path.join(tmp, f"w{world}_r{k}.json"))) for k in range(world)]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_reproduce_the_single_rank_run(cuda_device, tmp_path):
    one = _run(1, str(tmp_path))[0]
    two = _run(2, str(tmp_path))
    # generation: every sample's latents are identical whichever rank / batch produced them
    lat2 = {}
    for r in two:
        lat2.update(r["latents"])
    assert sorted(lat2) == sorted(one["latents"]) == ["0", "1", "2", "3"]
    for k in one["latents"]:
        assert lat2[k] == one["latents"][k], f"sample {k}: 2-rank latents differ from the 1-rank run"
    # training: allreduced gradient == mean of the two single-rank (per-shard) gradients; None stays None
    g0, g1 = one["grads"]["0"], one["grads"]["1"]
    for r in two:
        (got,) = r["grads"].values()
        for n in g0:
            parts = [x for x in (g0[n], g1[n]) if x is not None]
            if not parts:
                assert got[n] is None, n
                continue
            want = torch.tensor(parts, dtype=torch.float64).sum(0) / 2
            have = torch.tensor(got[n], dtype=torch.float64)
            # the two runs are separate processes: cuDNN autotuning may pick different (TF32) convolution algorithms for the
            # frozen backbone, so per-rank gradients agree to ~1e-3, not bitwise; a wrong reduction (sum instead of mean, a
            # dropped or doubled shard) is off by a factor
            err = (have - want).norm() / want.norm().clamp_min(1e-30)
            assert err <= 2e-2, f"{n}: relative error {err:.3e}"
