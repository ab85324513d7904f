"""Supervised evaluation calls on the CUDA path (pips_b200/supervised.py, csrc/score_loss.cu): the C entry points'
argument checks, and the two identities the score-loss kernels rest on, checked in torch on the CPU."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import pips_oracle as po
from pips_b200 import Pips, _lib as L, torch_path
from pips_b200.supervised import score_targets
from tests.golden.make_golden import LOSS_CASE, case_inputs, loss_targets


def test_score_loss_symbols_reject_bad_arguments_without_gpu():
    lib = L.load()
    for name in ("pips_score_grid", "pips_score_loss_scratch_floats", "pips_score_loss", "pips_score_loss_finalize"):
        assert name in L.EXPORTS
    assert lib.pips_score_grid(None, 16, 48, 64, None, None) != 0
    assert b"pips_score_grid: null pointer" in lib.pips_last_error()
    p = torch.zeros(1)
    lvl = L.ptr_array([p, p, p, p])
    assert lib.pips_score_grid(lvl, 0, 48, 64, L.ptr(p), None) != 0 and b"empty problem" in lib.pips_last_error()
    assert lib.pips_score_grid(lvl, 1, 4, 64, L.ptr(p), None) != 0 and b"too small" in lib.pips_last_error()
    assert lib.pips_score_loss(None, 1, 8, 4, 16, 16, None, None, 0, 4, 0, 1, None, None) != 0
    assert b"pips_score_loss: null pointer" in lib.pips_last_error()
    q = L.ptr(p)
    assert lib.pips_score_loss(q, 1, 8, 0, 16, 16, q, q, 0, 4, 0, 1, q, None) != 0 and b"empty problem" in lib.pips_last_error()
    assert lib.pips_score_loss(q, 1, 8, 4, 16, 16, q, q, 2, 4, 0, 1, q, None) != 0 and b"outside n_total" in lib.pips_last_error()
    assert lib.pips_score_loss(q, 1, 8, 4, 16, 16, q, q, 0, 4, 1, 1, q, None) != 0 and b"iteration" in lib.pips_last_error()
    assert lib.pips_score_loss_finalize(None, 32, 1, 16, 16, None, None, None) != 0
    assert b"pips_score_loss_finalize: null pointer" in lib.pips_last_error()
    assert lib.pips_score_loss_finalize(q, 0, 1, 16, 16, q, q, None) != 0 and b"empty problem" in lib.pips_last_error()
    assert lib.pips_score_loss_scratch_floats(0, 4, 48, 64) == 0
    # 3072 pixels = 24 blocks of 128 negatives + 1 positive per (track, iteration), then fp64 block sums
    assert lib.pips_score_loss_scratch_floats(1000, 4, 48, 64) == 4 * 1000 * 25 + 6


def _dense_fcp(f, pyramid, H8, W8):
    """torch_path's order (nets/pips.py:384-398, :504-511): dot products per level, then upsample and sum."""
    B, S, N, C = f.shape
    vols = [torch.matmul(f, lv.flatten(3)).reshape(B, S, N, *lv.shape[-2:]) / math.sqrt(C) for lv in pyramid]
    return sum(F.interpolate(v.flatten(0, 1), (H8, W8), mode="bilinear", align_corners=True).reshape(B, S, N, H8, W8)
               for v in vols)


def test_grid_rewrite_equals_dense_score_maps():
    """<f, sum_l interp(F_l) / sqrt(C)> == sum_l interp(<f, F_l> / sqrt(C)) on the LOSS_CASE feature maps."""
    c = LOSS_CASE
    m = Pips(S=8, stride=c["stride"]).eval()
    m.load_state_dict(po.init_state_dict(seed=c["seed"], head_scale=c["head_scale"]), strict=True)
    rgbs, xys, _ = case_inputs(c)
    with torch.no_grad():
        fmaps = m.encode(rgbs, torch_only=True)                          # (B,S,128,H8,W8)
        B, S, C, H8, W8 = fmaps.shape
        pyramid = [fmaps]
        for _ in range(3):
            p = F.avg_pool2d(pyramid[-1].flatten(0, 1), 2, stride=2)
            pyramid.append(p.reshape(B, S, *p.shape[1:]))
        coords = (xys / c["stride"]).reshape(B, 1, -1, 2).repeat(1, S, 1, 1)
        f0 = torch_path.sample_clamped(fmaps[:, 0], coords[:, 0, :, 0], coords[:, 0, :, 1])
        f = f0.unsqueeze(1).repeat(1, S, 1, 1) + 0.3 * torch.randn(B, S, f0.shape[1], C, generator=torch.Generator().manual_seed(0))
        dense = _dense_fcp(f, pyramid, H8, W8)
        grid = sum(F.interpolate(lv.flatten(0, 1), (H8, W8), mode="bilinear", align_corners=True) for lv in pyramid)
        grid = grid.reshape(B, S, C, H8 * W8) / math.sqrt(C)
        rewrite = torch.matmul(f, grid).reshape(dense.shape)
    err = (rewrite - dense).abs().max().item()
    assert err <= 1e-5 * dense.abs().max().item(), (err, dense.abs().max().item())


def decomposed_ce(fcps, target):
    """The score loss as the kernels compute it: per (track, iteration) the sum of softplus(fcp) over the pixels other
    than the target and fcp at the target, then the fp64 reduction of pips_score_loss_finalize."""
    B, S, I, N, H8, W8 = fcps.shape
    fcp = fcps.permute(0, 1, 3, 2, 4, 5).reshape(B * S * N, I, H8 * W8).double()
    g = target.reshape(-1).long()
    kept = g >= 0
    fcp, g = fcp[kept], g[kept]
    at_g = fcp.gather(2, g.view(-1, 1, 1).expand(-1, I, 1)).squeeze(2)
    neg = F.softplus(fcp).sum(2) - F.softplus(at_g)
    k = kept.sum().item() * I
    return F.softplus(-at_g).sum() / (1e-6 + k) + neg.sum() / (1e-6 + k * (H8 * W8 - 1))


def _targets_with_every_exclusion(B, S, N, H8, W8, stride, seed):
    g = torch.Generator().manual_seed(seed)
    px = torch.rand(B, S, N, 2, generator=g) * torch.tensor([W8 + 4.0, H8 + 4.0]) - 2.0   # some outside the map
    px[..., 0, :] = torch.tensor([2.5, 3.5])                                              # x.5 ties: round half to even
    px[..., 1, :] = torch.tensor([W8 - 0.5, H8 - 0.5])                                    # rounds onto the border, or past it
    px[..., 2, :] = torch.tensor([-0.5, 0.5])
    vis = (torch.rand(B, S, N, generator=g) > 0.3).float()
    valids = (torch.rand(B, S, N, generator=g) > 0.2).float()
    return px * stride, vis, valids


@pytest.mark.parametrize("H8,W8", [(12, 16), (9, 13)])
def test_decomposition_equals_score_map_loss(H8, W8):
    B, S, I, N, stride = 2, 8, 3, 7, 4
    fcps = torch.randn(B, S, I, N, H8, W8, generator=torch.Generator().manual_seed(1)) * 8
    trajs, vis, valids = _targets_with_every_exclusion(B, S, N, H8, W8, stride, seed=H8)
    target = score_targets(trajs, vis, valids, stride, H8, W8)
    assert (target >= 0).any() and (target < 0).any()
    ref = torch_path.score_map_loss(fcps, trajs / float(stride), vis, valids)
    got = decomposed_ce(fcps, target)
    assert abs(got.item() - ref.item()) <= 1e-6 * abs(ref.item()), (got.item(), ref.item())
    # torch.round rounds half to even: 2.5 -> 2, 3.5 -> 4
    assert target[0, 0, 0].item() == (-1 if not (vis[0, 0, 0] > 0 and valids[0, 0, 0] > 0) else 4 * W8 + 2)


def test_decomposition_with_every_track_excluded_is_zero():
    B, S, I, N, H8, W8 = 1, 8, 2, 3, 8, 8
    fcps = torch.randn(B, S, I, N, H8, W8)
    trajs = torch.full((B, S, N, 2), 100.0)
    target = score_targets(trajs, torch.ones(B, S, N), torch.ones(B, S, N), 1, H8, W8)
    assert (target == -1).all()
    assert torch_path.score_map_loss(fcps, trajs, torch.ones(B, S, N), torch.ones(B, S, N)).item() == 0.0
    assert decomposed_ce(fcps, target).item() == 0.0


def test_cuda_setting_with_cpu_tensors_is_the_torch_path():
    c = LOSS_CASE
    sd = po.init_state_dict(seed=c["seed"], head_scale=c["head_scale"])
    rgbs, xys, _ = case_inputs(c)
    tg, vg, va = loss_targets(c, xys)
    out = []
    for mode in ("torch", "cuda"):
        m = Pips(S=8, stride=c["stride"], supervised=mode).eval()
        m.load_state_dict(sd, strict=True)
        with torch.no_grad():
            out.append(m(xys, rgbs, iters=1, trajs_g=tg, vis_g=vg, valids=va))
    assert torch.equal(out[0][0][0], out[1][0][0]) and torch.equal(out[0][2], out[1][2])
    assert all(torch.equal(a, b) for a, b in zip(out[0][3], out[1][3]))
    with pytest.raises(ValueError):
        Pips(S=8, stride=8, supervised="triton")
