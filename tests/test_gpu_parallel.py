"""Two-GPU NCCL test of parallel.sharded_infer with the real engine under torchrun (SURVEY.md 8e): every rank runs its
shard of the batch on its own replica; the stacked result on every rank equals the single-GPU result bit for bit (images
are independent; the per-image arithmetic does not depend on which rank runs it, only on the plan's batch size, so both
sides use per-rank batch 2).  Needs 2 GPUs; skipped on a machine with one."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["GP_ROOT"])
from genpercept_b200 import weights as W
from genpercept_b200.parallel import sharded_infer, shard_bounds
from genpercept_b200.pipeline import GenPerceptPipeline
rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
state = W.synth_state(1234, with_dpt=False)
te = torch.from_numpy(np.load(os.path.join(os.environ["GP_ROOT"], "tests", "golden", "empty_text_embed_2x1024.npy")).astype(np.float32))[None]
pipe = GenPerceptPipeline(unet=state["unet"], vae=state["vae"], text_embed=te, torch_dtype=torch.float16, device=local)
g = torch.Generator().manual_seed(3)
rgb = torch.randint(0, 256, (4, 3, 64, 96), generator=g, dtype=torch.uint8)
infer = lambda x: pipe.single_infer(x.cuda(), mode="depth")
full = sharded_infer(infer, rgb, stacked=True)
mine = sharded_infer(infer, rgb, stacked=False)
lo, hi = shard_bounds(4, dist.get_world_size(), rank)
single = torch.cat([infer(rgb[0:2]), infer(rgb[2:4])])          # the same per-call batch size as a shard
ok = tuple(full.shape) == (4, 1, 64, 96) and torch.equal(full, single) and torch.equal(mine, single[lo:hi])
print(f"rank {rank}: ok={bool(ok)} max|full-single|={(full - single).abs().max().item():.3e}", flush=True)
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 1)
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_infer_two_gpus_nccl(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", "29581", str(script)], capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, GP_ROOT=ROOT))
    print(p.stdout[-2000:])
    assert p.returncode == 0, p.stderr[-3000:]
    assert p.stdout.count("ok=True") == 2
