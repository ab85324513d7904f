"""Supervised evaluation calls on the CUDA path: ``Pips.forward(..., trajs_g=, vis_g=, valids=)`` under ``no_grad`` with
``is_train=False`` -- the validation step of ``train.py`` and the evaluations of ``test_on_flt.py`` / ``test_on_crohd.py``.

The refinement loop is the inference loop; the score-map loss (nets/pips.py:58-90) is computed next to it by
``csrc/score_loss.cu`` from the loop state, without the dense score maps ``fcps``.  The two small losses
(``sequence_loss``, the visibility ``balanced_ce_loss``) are the torch path's own functions applied to the CUDA outputs.
"""
from __future__ import annotations

import torch

from . import torch_path


def score_targets(trajs_g: torch.Tensor, vis_g: torch.Tensor, valids: torch.Tensor, stride: float, H8: int,
                  W8: int) -> torch.Tensor:
    """The one-hot targets of ``score_map_loss`` (nets/pips.py:58-90) as pixel indices: (B,S,N) int32 holding
    ``y*W8 + x`` of the rounded ground truth in feature-map pixels, or -1 where the loss leaves the track out."""
    xy = (trajs_g / float(stride)).round().long()          # torch.round: half to even, like the reference
    x, y = xy[..., 0], xy[..., 1]
    keep = (x >= 0) & (x <= W8 - 1) & (y >= 0) & (y <= H8 - 1) & (valids > 0) & (vis_g > 0)
    return torch.where(keep, y * W8 + x, torch.full_like(x, -1)).to(torch.int32).contiguous()


def forward_cuda(model, xys, rgbs, coords_init, feat_init, iters, trajs_g, vis_g, valids, return_feat):
    """``Pips.forward`` with ground truth, the refinement loop and the score-map loss on the GPU.  Trajectories, vis_e
    and ffeat are those of the same call without ground truth (the loss kernels only read the loop state)."""
    B, N, _ = xys.shape
    with torch.no_grad():
        fmaps = model.encode(rgbs)
        H8, W8 = fmaps.shape[-2:]
        target = score_targets(trajs_g.to(rgbs.device), vis_g.to(rgbs.device), valids.to(rgbs.device), model.stride,
                               H8, W8)
        preds, preds2, vis_e, ffeat, ce = model._refine(xys, fmaps, coords_init, feat_init, iters, score_target=target)
        losses = (torch_path.sequence_loss(preds, trajs_g, vis_g, valids, 0.8),
                  torch_path.balanced_ce_loss(vis_e, vis_g, valids)[0], ce)
    if return_feat:
        return preds, preds2, vis_e, ffeat, losses
    return preds, preds2, vis_e, losses
