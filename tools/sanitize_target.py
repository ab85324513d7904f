"""Tiny end-to-end run for compute-sanitizer: one forward of the smallest parity configuration (128x160 clip, 24
particles, 2 iterations, eager launches -- no CUDA graph) through every kernel of the hot path: fnet (conv_tc, inorm,
resize, stem), pyramid, init gather, corr_gather, gemm_tc / gemm_tc2, tokenmix_tc, ln_pool, update, vis head, and one
supervised evaluation call (score grid, score loss, finalize).
With WORLD_SIZE=2 (torchrun) it runs the particle-sharded path: peer-slab stores, pips_peer_scatter, pips_peer_barrier."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("PIPS_B200_GRAPH", "0")
from pips_b200 import synthetic  # noqa: E402

world = int(os.environ.get("WORLD_SIZE", "1"))
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=dev)
model = synthetic.seeded_model(stride=8, seed=1).to(dev).eval()
if world > 1:
    model.shard_particles()
rgbs = synthetic.smooth_video(1, 8, 128, 160, seed=11).to(dev)
xys = synthetic.random_queries(1, 24, 128, 160, seed=12).to(dev)
xys[0, 0] = torch.tensor([-4.0, 3.0], device=dev)                 # out-of-bounds query: zero-filled TMA boxes
with torch.no_grad():
    for _ in range(2):                                            # second call: slab / buffer reuse
        preds, _, vis, _ = model(xys, rgbs, iters=2)
    big = synthetic.random_queries(1, 300, 128, 160, seed=13).to(dev)   # 2400 rows: the CTA-pair GEMM and its tail tiles
    p2 = model(big, rgbs, iters=1)[0]
    if world == 1:                                                # supervised evaluation call: the score-loss kernels
        model.supervised = "cuda"
        g = torch.Generator().manual_seed(14)
        tg = (xys.cpu()[:, None] + torch.randn(1, 8, 24, 2, generator=g) * 4).to(dev)
        vg = (torch.rand(1, 8, 24, generator=g) > 0.3).float().to(dev)
        losses = model(xys, rgbs, iters=2, trajs_g=tg, vis_g=vg, valids=torch.ones_like(vg))[3]
        assert all(bool(torch.isfinite(l)) for l in losses)
torch.cuda.synchronize()
print("sanitize target ok: finite =", bool(torch.isfinite(preds[-1]).all() and torch.isfinite(vis).all() and torch.isfinite(p2[-1]).all()),
      "kernels launched per forward =", model.engine.launches)
if world > 1:
    model.close_peer_slabs()
    dist.destroy_process_group()
