"""Supervised evaluation calls on the CUDA path (Pips(supervised='cuda'), csrc/score_loss.cu) against the reference's
recorded losses, the torch path on the same GPU and dense fp32 torch computations (B200 only)."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import pips_oracle as po
from pips_b200 import Pips, _lib as L, torch_path
from pips_b200.supervised import score_targets
from tests.golden.make_golden import LOSS_CASE, case_inputs, loss_targets

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_outputs.npz"))


def _model(stride=LOSS_CASE["stride"], seed=LOSS_CASE["seed"], **kw):
    m = Pips(S=8, stride=stride, **kw).to(DEV).eval()
    m.load_state_dict(po.init_state_dict(seed=seed, head_scale=LOSS_CASE["head_scale"]), strict=True)
    return m


def _loss_case():
    c = LOSS_CASE
    rgbs, xys, _ = case_inputs(c)
    tg, vg, va = loss_targets(c, xys)
    return rgbs.to(DEV), xys.to(DEV), tg.to(DEV), vg.to(DEV), va.to(DEV)


# strict mode meets the CPU torch path's rtol 1e-4.  Default mode (fnet on the tcgen05 convolutions, bf16x3 mixer GEMMs):
# measured on a B200, largest relative error 2.0e-6 (vis_loss); the tolerance is 10x that.
@pytest.mark.parametrize("mode,rtol", [("strict", 1e-4), ("default", 2e-5)])
def test_losses_match_reference(mode, rtol):
    kw = dict(precision="fp32", fnet_mode="plain") if mode == "strict" else {}
    m = _model(supervised="cuda", **kw)
    rgbs, xys, tg, vg, va = _loss_case()
    with torch.no_grad():
        preds, preds2, vis_e, losses = m(xys, rgbs, iters=LOSS_CASE["iters"], trajs_g=tg, vis_g=vg, valids=va)
    assert len(preds2) == LOSS_CASE["iters"] + 4
    assert np.abs(torch.stack(preds).cpu().numpy() - GOLD["loss_s8/preds"]).max() < 1e-3
    assert np.abs(vis_e.cpu().numpy() - GOLD["loss_s8/vis_e"]).max() < 2e-3
    assert all(l.dim() == 0 and l.is_cuda for l in losses)
    got = np.array([float(l) for l in losses])
    ref = GOLD["loss_s8/losses"]
    print(f"losses [{mode}]: {got} vs {ref}, rel err {np.abs(got - ref) / np.abs(ref)}")
    assert np.allclose(got, ref, rtol=rtol, atol=1e-5), (got, ref)


def _exclusion_targets(B, N, H, W, stride, xys, seed):
    """Ground truth with every case score_map_loss excludes: outside the map, x.5 ties, invalid, invisible."""
    g = torch.Generator().manual_seed(seed)
    tg = xys.cpu()[:, None] + torch.cumsum(torch.randn(B, 8, N, 2, generator=g) * 3, 1)
    tg[:, :, 0] = torch.tensor([-3.0 * stride, 5.0 * stride])
    tg[:, :, 1] = torch.tensor([W + 2.0 * stride, 4.0 * stride])
    tg[:, :, 2] = torch.tensor([2.5 * stride, 3.5 * stride])
    vg = (torch.rand(B, 8, N, generator=g) > 0.3).float()
    va = (torch.rand(B, 8, N, generator=g) > 0.1).float()
    return tg.to(DEV), vg.to(DEV), va.to(DEV)


@pytest.mark.parametrize("H,W,stride,N", [(384, 512, 8, 300), (384, 512, 4, 300), (128, 200, 8, 37)])
def test_losses_match_torch_path_on_gpu(H, W, stride, N):
    """384x512 gives 48x64 / 96x128 maps (multiples of the 256-pixel tile); 128x200 at stride 8 gives 16x25 = 400."""
    B, iters = 2, 4
    rgbs = po.smooth_video(B, 8, H, W, seed=31).to(DEV)
    xys = po.random_queries(B, N, H, W, seed=32).to(DEV)
    tg, vg, va = _exclusion_targets(B, N, H, W, stride, xys, seed=33)
    out = {}
    for mode in ("torch", "cuda"):
        m = _model(stride=stride, supervised=mode, precision="fp32", fnet_mode="plain")
        with torch.no_grad():
            out[mode] = m(xys, rgbs, iters=iters, trajs_g=tg, vis_g=vg, valids=va)
    got = np.array([float(l) for l in out["cuda"][3]])
    ref = np.array([float(l) for l in out["torch"][3]])
    print(f"{H}x{W}/{stride}: cuda {got} torch {ref} rel {np.abs(got - ref) / np.abs(ref)}")
    assert np.allclose(got, ref, rtol=1e-4, atol=1e-5), (got, ref)


def _run(m, xys, rgbs, **kw):
    with torch.no_grad():
        p, _, v, f, losses = m(xys, rgbs, iters=3, return_feat=True, **kw)
    return torch.stack(p), v, f, losses


@pytest.mark.parametrize("graph", [True, False])
def test_trajectories_unchanged_and_runs_repeat(graph):
    rgbs, xys, tg, vg, va = _loss_case()
    m = _model(supervised="cuda")
    m.engine.use_graph = graph                         # what PIPS_B200_GRAPH=0 selects
    plain = _run(m, xys, rgbs)
    sup = _run(m, xys, rgbs, trajs_g=tg, vis_g=vg, valids=va)
    again = _run(m, xys, rgbs, trajs_g=tg, vis_g=vg, valids=va)
    assert plain[3] is None
    for a, b in zip(plain[:3], sup[:3]):
        assert torch.equal(a, b)
    for a, b in zip(sup[3], again[3]):
        assert torch.equal(a, b)


def test_chunked_losses_are_bit_identical():
    rgbs, xys, tg, vg, va = _loss_case()
    one = _run(_model(supervised="cuda"), xys, rgbs, trajs_g=tg, vis_g=vg, valids=va)
    chunked = _run(_model(supervised="cuda", max_seqs=8), xys, rgbs, trajs_g=tg, vis_g=vg, valids=va)  # 4 particles per chunk
    for a, b in zip(one[:3], chunked[:3]):
        assert torch.equal(a, b)
    for a, b in zip(one[3], chunked[3]):
        assert torch.equal(a, b)


def test_other_supervised_calls_stay_on_the_torch_path():
    rgbs, xys, tg, vg, va = _loss_case()
    calls = []
    real = torch_path.score_map_loss

    def spy(*a, **k):
        calls.append(1)
        return real(*a, **k)

    class Saver:
        save_this = True

    cuda = _model(supervised="cuda")
    cases = [(cuda, dict(), True), (cuda, dict(is_train=True), False), (cuda, dict(sw=Saver()), False),
             (_model(), dict(), False)]
    torch_path.score_map_loss = spy
    try:
        for m, kw, grad in cases:
            n = len(calls)
            with torch.set_grad_enabled(grad):
                m(xys, rgbs, iters=1, trajs_g=tg, vis_g=vg, valids=va, **kw)
            assert len(calls) == n + 1, kw
        n = len(calls)
        with torch.no_grad():
            cuda(xys, rgbs, iters=1, trajs_g=tg, vis_g=vg, valids=va)
        assert len(calls) == n                                 # the CUDA route never builds the dense score maps
    finally:
        torch_path.score_map_loss = real


def test_peak_memory_holds_no_dense_score_maps():
    B, N, H, W, stride, iters = 2, 300, 384, 512, 8, 4
    rgbs = po.smooth_video(B, 8, H, W, seed=41).to(DEV)
    xys = po.random_queries(B, N, H, W, seed=42).to(DEV)
    tg, vg, va = _exclusion_targets(B, N, H, W, stride, xys, seed=43)

    def peak(**kw):
        """the first call of a fresh model: everything it allocates, the buffers its CUDA graphs keep included"""
        m = _model(stride=stride, supervised="cuda")
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        with torch.no_grad():
            m(xys, rgbs, iters=iters, **kw)
        torch.cuda.synchronize()
        p = torch.cuda.max_memory_allocated() - base
        del m
        torch.cuda.empty_cache()
        return p

    plain = peak()
    sup = peak(trajs_g=tg, vis_g=vg, valids=va)
    H8, W8 = H // stride, W // stride
    ppad = -(-H8 * W8 // L.SCORE_TILE) * L.SCORE_TILE
    allowed = 2 * B * 8 * ppad * 128 * 2 + 4 * L.load().pips_score_loss_scratch_floats(B * 8 * N, iters, H8, W8)
    dense = B * 8 * iters * N * H8 * W8 * 4
    print(f"peak: plain {plain / 2**20:.1f} MiB, supervised {sup / 2**20:.1f} MiB, grid + partials {allowed / 2**20:.1f} MiB, "
          f"dense score maps would be {dense / 2**20:.1f} MiB")
    assert sup - plain <= 1.1 * allowed


def _levels(frames, H8, W8, seed):
    g = torch.Generator().manual_seed(seed)
    f0 = torch.randn(frames, 128, H8, W8, generator=g)
    lv = [f0]
    for _ in range(3):
        lv.append(F.avg_pool2d(lv[-1], 2, stride=2))
    return lv


@pytest.mark.parametrize("H8,W8", [(16, 16), (20, 13)])
def test_score_kernels_against_dense_fp32(H8, W8):
    lib = L.load()
    B, S, N, iters = 1, 8, 5, 1
    frames = B * S
    lv = _levels(frames, H8, W8, seed=H8)
    lvl = [l.permute(0, 2, 3, 1).contiguous().to(DEV) for l in lv]
    ppad = -(-H8 * W8 // L.SCORE_TILE) * L.SCORE_TILE
    grid = torch.empty(2, frames, ppad, 128, dtype=torch.bfloat16, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    L.check(lib.pips_score_grid(L.ptr_array(lvl), frames, H8, W8, L.ptr(grid), st))
    ref = sum(F.interpolate(l, (H8, W8), mode="bilinear", align_corners=True) for l in lv) / math.sqrt(128)
    ref = ref.permute(0, 2, 3, 1).reshape(frames, H8 * W8, 128)
    gr = grid[0].float() + grid[1].float()
    assert (gr[:, :H8 * W8].cpu() - ref).abs().max().item() < 1e-5 * ref.abs().max().item() + 1e-6
    assert (grid[:, :, H8 * W8:] == 0).all()

    g = torch.Generator().manual_seed(7)
    ffeats = (torch.randn(B * N, S, 128, generator=g) * 2).to(DEV)
    tgt = torch.randint(0, H8 * W8, (B, S, N), generator=g, dtype=torch.int32)
    tgt[0, 1, 2] = -1
    tgt[0, 3, 0] = H8 * W8 - 1
    tgt = tgt.to(DEV)
    partial = torch.empty(lib.pips_score_loss_scratch_floats(B * S * N, iters, H8, W8), dtype=torch.float32, device=DEV)
    ce = torch.zeros(1, device=DEV)
    L.check(lib.pips_score_loss(L.ptr(grid), B, S, N, H8, W8, L.ptr(ffeats), L.ptr(tgt), 0, N, 0, iters, L.ptr(partial), st))
    L.check(lib.pips_score_loss_finalize(L.ptr(tgt), B * S * N, iters, H8, W8, L.ptr(partial), L.ptr(ce), st))
    torch.cuda.synchronize()

    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        f = ffeats.cpu().reshape(B, N, S, 128).permute(0, 2, 1, 3)               # (B,S,N,128)
        fcp = torch.matmul(f.reshape(frames, N, 128), ref.transpose(1, 2))        # (frames, N, P) dense fp32
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    rows = frames * N
    blocks = ppad // 128
    neg = partial[:rows * blocks].reshape(blocks, rows).cpu()
    pos = partial[rows * blocks:rows * (blocks + 1)].cpu()
    t = tgt.cpu().reshape(rows).long()
    fr = fcp.reshape(rows, H8 * W8)
    sp = F.softplus(fr.double())
    keep = t >= 0
    col = torch.arange(H8 * W8)
    for blk in range(blocks):
        m = ((col >= blk * 128) & (col < (blk + 1) * 128)).double()
        want = (sp * m).sum(1) - torch.where(keep & (t // 128 == blk), sp.gather(1, t.clamp(min=0).view(-1, 1)).squeeze(1), torch.zeros(rows, dtype=torch.float64))
        assert torch.allclose(neg[blk][keep].double(), want[keep], rtol=2e-5, atol=1e-3), blk
    want_pos = fr.gather(1, t.clamp(min=0).view(-1, 1)).squeeze(1)
    assert torch.allclose(pos[keep], want_pos[keep], rtol=1e-5, atol=2e-4)
    fcps = fcp.reshape(B, S, 1, N, H8, W8)
    trajs = torch.stack([t % W8, t // W8], -1).float().reshape(B, S, N, 2)
    vis = keep.float().reshape(B, S, N)
    want_ce = torch_path.score_map_loss(fcps, trajs, vis, torch.ones(B, S, N))
    assert abs(ce.item() - want_ce.item()) <= 1e-5 * abs(want_ce.item())
    assert torch.equal(score_targets(trajs * 4, vis, torch.ones(B, S, N), 4, H8, W8), torch.where(keep, t, -1).int().reshape(B, S, N))
