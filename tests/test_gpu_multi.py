"""GPU, >= 2 devices: GradBuckets over NCCL with the three-stream hot-path step (gradients of one bucket accumulated on
different streams), against a single-process run over the concatenated batch.  Skipped on single-GPU machines; run on
one with two or more GPUs with `python -m pytest tests/test_gpu_multi.py -m gpu`."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import json, os, sys
sys.path.insert(0, %(root)r)
import torch, torch.distributed as dist
from robust_e2e_gan_b200.parallel import GradBuckets, init_distributed
from robust_e2e_gan_b200.hotpath import HotPath, make_batch
rank, world = init_distributed()
dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
torch.cuda.set_device(dev)
cfg = dict(B=4, T=64, F=257, M=40, Th=16, D=320, A=320, Z=300, C=10, filts=100, V=97, U=5, steps=6)
hp = HotPath(cfg, seed=3, overlap=True).to(dev)               # identical init on every rank
buckets = GradBuckets(hp.trainable(), bucket_mb=0.5)           # several buckets; ctc_lo / att parameters mixed
res = []
for step in range(2):
    b = make_batch(cfg, seed=100 + rank).to(dev)
    buckets.zero()
    hp.step(b)
    buckets.finish()
    torch.cuda.synchronize()
    res.append({k: p.grad.detach().double().cpu() for k, p in hp.named_parameters() if p.requires_grad})
# truth: mean over the ranks of single-rank gradients, each computed without buckets on this rank's device
truth = None
for r in range(world):
    hp2 = HotPath(cfg, seed=3, overlap=False).to(dev)
    out = hp2.step(make_batch(cfg, seed=100 + r).to(dev))
    g = {k: p.grad.detach().double().cpu() for k, p in hp2.named_parameters() if p.requires_grad}
    truth = g if truth is None else {k: truth[k] + g[k] for k in g}
truth = {k: v / world for k, v in truth.items()}
worst = 0.0
for k in truth:
    if k.endswith("gvec.bias"):
        continue
    scale = float(truth[k].abs().max()) or 1.0
    worst = max(worst, float((res[1][k] - truth[k]).abs().max()) / scale)
print(json.dumps({"rank": rank, "worst": worst, "nbuckets": len(buckets.buckets)}), flush=True)
dist.barrier()
dist.destroy_process_group()
'''


def test_grad_buckets_nccl_with_three_stream_step(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER % {"root": ROOT})
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29611", str(script)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    import re
    lines = [json.loads(m) for m in re.findall(r"\{[^{}]*\}", r.stdout)]
    assert len(lines) == 2 and all(l["nbuckets"] > 1 for l in lines)
    assert all(l["worst"] < 1e-5 for l in lines), lines
