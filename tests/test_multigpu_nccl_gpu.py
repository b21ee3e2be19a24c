"""N = 2 over NCCL (needs two GPUs: `python -m pytest tests/test_multigpu_nccl_gpu.py -m gpu` on a machine with two):
the gathered post-NMS records of two image shards of ONE global batch equal the single-GPU records (SURVEY.md §8(e))."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, %r)
from posecnn_b200 import parallel, synth
from posecnn_b200.networks.vgg16_convs import vgg16_convs, GraphedForward
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
B, H, W, C = 8, 96, 128, 6
net = vgg16_convs(num_classes=C, device=dev).init_random(seed=0, bias_std=0.05)
rgb, _ = synth.make_images(B, H, W, seed=9)
data = torch.from_numpy(rgb).to(dev)
meta = torch.from_numpy(np.stack([synth.make_meta(synth.intrinsics(H, W))] * B)).to(dev)
ext = torch.from_numpy(synth.extents_for(C)).to(dev)
whole = parallel.compact_records(parallel.pack_detections(net.forward(data, meta, ext, sync_rois=False, dense_vertex=False)))
o, n = parallel.shard_range(B, rank, world)
fwd = GraphedForward(net, data[o:o + n], meta[o:o + n], ext, pack_records=True, dense_vertex=False, batch_global=B, batch_offset=o)
pipe = parallel.GatherPipeline(world, fwd.layers["records"])
ok = True
for step in range(4):                      # the double-buffered pipeline, several steps in flight
    pipe.before_step()
    L = fwd(data[o:o + n])
    i = pipe.submit(L["records"])
    got = parallel.compact_records(pipe.results(i))
    ok = ok and torch.equal(got, whole)
pipe.drain()
torch.cuda.synchronize()
assert whole.shape[0] >= 2 and ok, (rank, whole.shape)
dist.barrier()
dist.destroy_process_group()
print("RANK_OK", rank, whole.shape[0])
''' % ROOT


def test_two_rank_gather_equals_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", str(port), str(script)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.count("RANK_OK") == 2, (out.stdout[-2000:], out.stderr[-3000:])


TRAIN_WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, %r)
from posecnn_b200 import parallel, synth
from posecnn_b200.networks.vgg16_convs import vgg16_convs
from posecnn_b200.train import Trainer
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
B, H, W, C = 4, 64, 96, 6
def problem():
    net = vgg16_convs(num_classes=C, device=dev, is_train=True, fold_vertex_head=False).init_random(seed=0, bias_std=0.02)
    net.params["score/weights"] *= 0.02; net.params["vertex_pred/weights"] *= 0.02; net.params["fc8/weights"] *= 0.01
    net.prepare()
    return net
rgb, _ = synth.make_images(B, H, W, seed=3)
sc = synth.make_scene(batch=B, height=H, width=W, num_classes=C, objects_per_image=3, seed=11, min_pixels=200)
centers = np.zeros((B, C, 3), np.float32)
for (b, cls, cx, cy, z) in sc["centers"]:
    centers[b, cls] = (cx, cy, z)
T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
data, gt, cen, meta, ext, gtp = T(rgb), T(sc["label"]), T(centers), T(sc["meta"].reshape(B, 48)), T(sc["extents"]), T(sc["gt"])
pts, sym = T(synth.make_model_points(C, 300)), torch.zeros(C, device=dev)
single = Trainer(problem(), lr=0.01, world=1)
ref = single.step(data, gt, cen, meta, ext, gtp, pts, sym)
o, n = parallel.shard_range(B, rank, world)
tr = Trainer(problem(), lr=0.01, world=world)
out = tr.step(data[o:o + n], gt[o:o + n], cen[o:o + n], meta[o:o + n], ext, gtp, pts, sym, batch_global=B, batch_offset=o)
torch.cuda.synchronize()
worst = 0.0
for name, g in out["grads"].items():
    w = ref["grads"][name]
    e = ((g - w).norm() / w.norm().clamp(min=1e-20)).item()
    worst = max(worst, e)
    assert e < 2e-3, (name, e)
for name in tr.master:
    assert torch.allclose(tr.master[name], single.master[name], rtol=1e-4, atol=1e-6), name
tot = torch.stack([out["loss_cls"][0], out["loss_vertex"][0], out["loss_pose"][0]])
dist.all_reduce(tot)
want = torch.stack([ref["loss_cls"][0], ref["loss_vertex"][0], ref["loss_pose"][0]])
assert torch.allclose(tot, want, rtol=1e-4, atol=1e-6), (tot, want)
dist.barrier()
dist.destroy_process_group()
print("TRAIN_RANK_OK", rank, worst)
''' % ROOT


def test_two_rank_training_step_equals_single_gpu(tmp_path):
    """configs[4] contract: one SGD step on image shards over 2 ranks (global loss normalisers, NCCL all-reduce of the gradients)
    == the step on the whole batch on one GPU (gradients to 2e-3 relative: only the fp32 summation order differs)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "train_worker.py"
    script.write_text(TRAIN_WORKER)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", str(port), str(script)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and out.stdout.count("TRAIN_RANK_OK") == 2, (out.stdout[-2000:], out.stderr[-3000:])
