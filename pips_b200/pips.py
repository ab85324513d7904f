"""Drop-in for the reference's ``nets.pips.Pips`` (nets/pips.py:400-611).

Same constructor, same ``forward(xys, rgbs, coords_init, feat_init, iters, trajs_g, vis_g, valids,
sw, return_feat, is_train)`` signature and return tuples, same ``state_dict`` keys -- so ``demo.py``,
``chain_demo.py``, ``test_on_*.py`` and ``saverloader.load`` work unchanged -- but at inference the
per-iteration refinement loop (nets/pips.py:459-559) runs in hand-written sm_100a CUDA
(libpips_b200.so) instead of ~150 eager torch ops per iteration, and the all-pairs correlation
volume is never materialised.

Extra, optional knobs (keyword-only; the reference signature is unchanged):
  precision   'bf16x3' (default; tcgen05 with hi/lo-split bf16 operands, fp32-class accuracy, meets
              the 1e-3 px parity target), 'bf16' (fast, ~1e-2 px), 'fp32' (CUDA-core GEMMs, exact)
  feat_dtype  'fp32' (default) or 'bf16' storage of the correlation pyramid
  fnet_mode   'tc' (default; residual stages and head as tcgen05 implicit-GEMM convolutions with bf16x3
              operands, element-wise stages fused, channels-last), 'fast' (cuDNN TF32 tensor-core
              convolutions over hi/lo-split operands instead), 'x3' (the same cuDNN convolutions through
              eager torch ops) or 'plain' (strict fp32 cuDNN)
  supervised  'torch' (default) or 'cuda': where a supervised evaluation call runs -- ground truth given, is_train=False,
              gradients off, no summary to save, CUDA inputs, not particle-sharded, not an nn.DataParallel replica.
              'cuda' runs it on the inference kernels and computes the score-map loss without the dense score maps
              (pips_b200/supervised.py; that loss is always bf16x3 on the tensor cores, whatever ``precision`` says).
              Every other supervised or training call stays on the torch path (torch_path.py).
Environment overrides: PIPS_B200_PRECISION, PIPS_B200_FEAT, PIPS_B200_FNET, PIPS_B200_SUPERVISED.
"""
from __future__ import annotations

import contextlib
import os
from typing import Optional

import torch
import torch.nn as nn

from .encoder import Encoder
from .engine import RefineEngine

LATENT = 128
CORR_LEVELS = 4
CORR_RADIUS = 3


class PreNormResidual(nn.Module):
    def __init__(self, dim: int, fn: nn.Module):
        super().__init__()
        self.fn = fn
        self.norm = nn.LayerNorm(dim)

    def forward(self, x):
        return self.fn(self.norm(x)) + x


class _MeanOverFrames(nn.Module):
    def forward(self, x):                      # (R, S, C) -> (R, C)
        return x.mean(dim=1)


def _feed_forward(dim: int, dense) -> nn.Sequential:
    # indices 0 and 3 carry the parameters, like the reference's FeedForward (nets/pips.py:102-109);
    # the Dropout(0.) slots are identities
    return nn.Sequential(dense(dim, dim * 4), nn.GELU(), nn.Identity(), dense(dim * 4, dim), nn.Identity())


def _conv1(cin, cout):
    return nn.Conv1d(cin, cout, kernel_size=1)


class DeltaBlock(nn.Module):
    """MLP-Mixer over the S x 519 token stack of one track (nets/pips.py:283-311, :111-123)."""

    def __init__(self, input_dim=LATENT, corr_levels=CORR_LEVELS, corr_radius=CORR_RADIUS, S=8, dim=512, depth=12):
        super().__init__()
        self.input_dim, self.S = input_dim, S
        kitchen = corr_levels * (2 * corr_radius + 1) ** 2 + input_dim + 64 * 3 + 3
        blocks = [nn.Sequential(PreNormResidual(dim, _feed_forward(S, _conv1)),
                                PreNormResidual(dim, _feed_forward(dim, nn.Linear))) for _ in range(depth)]
        self.to_delta = nn.Sequential(nn.Linear(kitchen, dim), *blocks, nn.LayerNorm(dim), _MeanOverFrames(),
                                      nn.Linear(dim, S * (input_dim + 2)))

    def forward(self, x):                      # x: (R, S, 519) already concatenated
        return self.to_delta(x).reshape(x.shape[0], self.S, self.input_dim + 2)


@contextlib.contextmanager
def _conv_math(allow_tf32: bool):
    """Pin cuDNN's conv math for fnet.  torch enables plain TF32 convolutions by default on Ampere+, which
    alone moves trajectories by ~1e-2 px (measured: fmaps error 2.5e-2); fnet therefore runs either in
    strict fp32 ('plain') or in the 3xTF32 split mode ('x3', fp32-class accuracy on the tensor cores)."""
    c, m = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        yield
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = c, m


class Pips(nn.Module):
    def __init__(self, S=8, stride=8, *, precision: Optional[str] = None, feat_dtype: Optional[str] = None,
                 fnet_mode: Optional[str] = None, max_seqs: int = 32768, supervised: Optional[str] = None):
        super().__init__()
        self.S = S
        self.stride = stride
        self.hidden_dim = 256
        self.latent_dim = LATENT
        self.corr_levels = CORR_LEVELS
        self.corr_radius = CORR_RADIUS

        self.fnet = Encoder(output_dim=LATENT, stride=stride)
        self.delta_block = DeltaBlock(input_dim=LATENT, corr_levels=CORR_LEVELS, corr_radius=CORR_RADIUS, S=S)
        self.norm = nn.GroupNorm(1, LATENT)
        self.ffeat_updater = nn.Sequential(nn.Linear(LATENT, LATENT), nn.GELU())
        self.vis_predictor = nn.Sequential(nn.Linear(LATENT, 1))

        precision = precision or os.environ.get("PIPS_B200_PRECISION", "bf16x3")
        feat_dtype = feat_dtype or os.environ.get("PIPS_B200_FEAT", "fp32")
        self._engine = RefineEngine(precision=precision, feat_dtype=feat_dtype, max_seqs=max_seqs)
        self._shard = None                      # (rank, world, group) when particle-sharded
        self.shard_fnet = True                  # sharded runs also split the encoder's frames over the ranks
        self.fnet_mode = fnet_mode or os.environ.get("PIPS_B200_FNET", "tc")
        if self.fnet_mode not in ("tc", "fast", "x3", "plain"):
            raise ValueError("fnet_mode must be 'tc' (tcgen05 implicit-GEMM convolutions, bf16x3), 'fast' (cuDNN 3xTF32 "
                             "convolutions, channels-last, fused element-wise kernels), 'x3' (3xTF32 convolutions through "
                             "eager torch ops) or 'plain' (strict fp32 cuDNN)")
        self.supervised = supervised or os.environ.get("PIPS_B200_SUPERVISED", "torch")
        if self.supervised not in ("torch", "cuda"):
            raise ValueError("supervised must be 'torch' (supervised calls on the differentiable torch path) or 'cuda' "
                             "(evaluation calls on the CUDA kernels, score-map loss without dense score maps)")

    # ------------------------------------------------------------------ configuration
    @property
    def engine(self) -> RefineEngine:
        return self._engine

    def shard_particles(self, group=None, balance: Optional[bool] = None) -> "Pips":
        """Particle-axis data parallelism (SURVEY.md section 8e): every rank owns a share of the tracks and a
        full copy of the feature pyramid; results are exchanged so each rank returns the full
        result.  Call after ``torch.distributed.init_process_group``.
        ``balance`` (default off; PIPS_B200_BALANCE=1 turns it on): after a few forwards the shares become proportional to
        each GPU's measured speed (sharding._Balance).  Measured on 8 B200s (profiles/r02_diag_8gpu.txt): under the power
        cap a GPU's speed drifts by +-3-5 % from step to step and WHICH GPU is slowest changes between runs, so a share
        fixed from a few samples does not beat equal shares -- kept as an option for boxes with a persistently slow GPU.
        Results do not depend on the shares (tracks are independent): bit-exact either way (tools/check_sharded.py)."""
        import torch.distributed as dist
        self._shard = (dist.get_rank(group), dist.get_world_size(group), group)
        if balance is None:
            balance = os.environ.get("PIPS_B200_BALANCE", "0") == "1"
        if balance and self._shard[1] > 1:
            from .sharding import _Balance
            self._balance = _Balance()
        else:
            self._balance = None
        return self

    def close_peer_slabs(self) -> None:
        """Collective: release the peer-mapped slabs of a particle-sharded model (results and feature maps).  They are
        re-created on demand by the next sharded forward."""
        for name in ("_peer_slab", "_fmap_peer_slab"):
            slab = getattr(self, name, None)
            if slab is not None:
                slab.close()
                setattr(self, name, None)
        self._engine.invalidate(graphs_only=True)

    # ------------------------------------------------------------------ forward
    def encode(self, rgbs: torch.Tensor, torch_only: bool = False) -> torch.Tensor:
        """nets/pips.py:436-445: normalise to [-1,1], fnet per frame -> (B,S,128,H8,W8) fp32.
        ``torch_only``: the plain torch module with strict-fp32 cuDNN math -- what the supervised / training path
        (torch_path.forward_torch) uses: it may run on nn.DataParallel replicas from worker threads (train.py:254),
        where per-parameter-pointer graph caches would be re-captured on every call and stream capture is unsafe."""
        B, S, C, H, W = rgbs.shape
        # the split paths detach the weights: inference only (the training path keeps plain cuDNN + autograd)
        infer = rgbs.is_cuda and not torch.is_grad_enabled() and not torch_only
        H8, W8 = H // self.stride, W // self.stride
        if self.fnet_mode == "tc" and infer:
            from .encoder_fast import fnet_tc, fnet_tc_graphed
            raw = rgbs if rgbs.dtype in (torch.float32, torch.bfloat16) else rgbs.float()
            run = fnet_tc_graphed if self._engine.use_graph else fnet_tc
            f = run(self.fnet, raw.reshape(B * S, C, H, W).contiguous())  # normalisation fused into the stem
            return f.reshape(B, S, H8, W8, self.latent_dim).permute(0, 1, 4, 2, 3)   # logical (B,S,128,H8,W8)
        x = 2 * (rgbs.float() / 255.0) - 1.0
        if self.fnet_mode == "fast" and infer:
            from .encoder_fast import fnet_fast
            with _conv_math(allow_tf32=True):
                f = fnet_fast(self.fnet, x.reshape(B * S, C, H, W))       # (B*S, H8, W8, 128) NHWC
            return f.reshape(B, S, H8, W8, self.latent_dim).permute(0, 1, 4, 2, 3)  # logical (B,S,128,H8,W8)
        x3 = self.fnet_mode in ("x3", "fast", "tc") and infer
        self.fnet.mode = "x3" if x3 else "plain"
        with _conv_math(allow_tf32=x3):
            fmaps = self.fnet(x.reshape(B * S, C, H, W))
        return fmaps.reshape(B, S, self.latent_dim, H8, W8)

    def forward(self, xys, rgbs, coords_init=None, feat_init=None, iters=3, trajs_g=None, vis_g=None, valids=None,
                sw=None, return_feat=False, is_train=False):
        B, N, D = xys.shape
        assert (D == 2)
        B, S, C, H, W = rgbs.shape

        save = sw is not None and getattr(sw, "save_this", False)
        if (trajs_g is not None and self.supervised == "cuda" and not is_train and not torch.is_grad_enabled() and not save
                and rgbs.is_cuda and self._shard is None and not getattr(self, "_is_replica", False)):
            if N == 0:
                raise RuntimeError("pips_b200.Pips: no particles (xys has N = 0); the reference raises here as well")
            from .supervised import forward_cuda
            return forward_cuda(self, xys, rgbs, coords_init, feat_init, iters, trajs_g, vis_g, valids, return_feat)
        slow = trajs_g is not None or is_train or save
        if slow:
            from .torch_path import forward_torch
            return forward_torch(self, xys, rgbs, coords_init=coords_init, feat_init=feat_init, iters=iters,
                                 trajs_g=trajs_g, vis_g=vis_g, valids=valids, sw=sw, return_feat=return_feat,
                                 is_train=is_train)
        if N == 0:
            # the reference fails on an empty particle axis (F.interpolate of the empty correlation volume,
            # nets/pips.py:509 -> RuntimeError; recorded in tests/golden as edge/n0_error): same error type here
            raise RuntimeError("pips_b200.Pips: no particles (xys has N = 0); the reference raises here as well")
        if not rgbs.is_cuda:
            raise RuntimeError("pips_b200.Pips: the inference path is CUDA-only (sm_100a); move the model and "
                               "inputs to a CUDA device. There is no CPU fallback.")
        with torch.no_grad():
            if self._shard is not None and self._shard[1] > 1 and self.shard_fnet and self.fnet_mode == "tc":
                from .sharding import encode_sharded
                fmaps = encode_sharded(self, rgbs)
            else:
                fmaps = self.encode(rgbs)
            return self.refine(xys, fmaps, coords_init=coords_init, feat_init=feat_init, iters=iters,
                               return_feat=return_feat)

    @torch.no_grad()
    def score_maps(self, xys, rgbs, particles, iters=3, coords_init=None, feat_init=None):
        """The dense score maps ``fcps`` of nets/pips.py:504-511,:565 for the chosen ``particles`` only
        (SURVEY.md section 8f-3): (B,S,iters,len(particles),H8,W8), i.e. ``fcps[:, :, :, particles]`` of the
        reference, without the all-pairs volume.  The reference's own consumers look at one particle
        (``fcps[0:1,:,:,0:1]``, nets/pips.py:572).  Also returns (coord_predictions, vis_e) of the same run."""
        if not rgbs.is_cuda:
            raise RuntimeError("pips_b200.Pips.score_maps is CUDA-only (sm_100a)")
        B, N, D = xys.shape
        assert (D == 2)
        S = rgbs.shape[1]
        fmaps = self.encode(rgbs)
        stride = float(self.stride)
        if coords_init is None:
            coords = (xys.detach().float() / stride).reshape(B, 1, N, 2).repeat(1, S, 1, 1)
        else:
            coords = coords_init.detach().float() / stride
        sel = torch.as_tensor(particles, dtype=torch.int64, device=rgbs.device).flatten()
        H8, W8 = fmaps.shape[-2:]
        fcps = torch.empty(B, S, iters, sel.numel(), H8, W8, dtype=torch.float32, device=rgbs.device)
        preds, vis_e, _ = self._engine.refine(self, fmaps.float(), coords,
                                              None if feat_init is None else feat_init.detach().float(), iters, stride,
                                              heat_sel=sel, heat_out=fcps)
        return fcps, [preds[i] for i in range(iters)], vis_e

    def refine(self, xys, fmaps, coords_init=None, feat_init=None, iters=3, return_feat=False):
        """Everything after fnet (nets/pips.py:450-611) given precomputed feature maps."""
        coord_predictions, coord_predictions2, vis_e, ffeat, _ = self._refine(xys, fmaps, coords_init, feat_init, iters)
        losses = None
        if return_feat:
            return coord_predictions, coord_predictions2, vis_e, ffeat, losses
        return coord_predictions, coord_predictions2, vis_e, losses

    def _refine(self, xys, fmaps, coords_init, feat_init, iters, score_target=None):
        """refine() as (coord_predictions, coord_predictions2, vis_e, ffeat, ce); ``score_target`` (B,S,N) int32
        (supervised.score_targets) also computes the score-map loss ``ce``, else ce is None."""
        B, N, _ = xys.shape
        S = fmaps.shape[1]
        stride = float(self.stride)
        xys_ = xys.detach().float() / stride                                            # :450
        if coords_init is None:
            coords = xys_.reshape(B, 1, N, 2).repeat(1, S, 1, 1)                        # :453
        else:
            coords = coords_init.detach().float() / self.stride                         # :455
        if feat_init is not None:
            feat_init = feat_init.detach().float()

        ce = None
        if score_target is not None:
            preds, vis_e, ffeat, ce = self._engine.refine(self, fmaps.float(), coords, feat_init, iters, stride,
                                                          score_target=score_target)
        elif self._shard is None or self._shard[1] == 1:
            preds, vis_e, ffeat = self._engine.refine(self, fmaps.float(), coords, feat_init, iters, stride)
        else:
            from .sharding import refine_sharded
            preds, vis_e, ffeat = refine_sharded(self, fmaps.float(), coords, feat_init, iters, stride)

        start = coords * stride
        coord_predictions = [preds[i] for i in range(iters)]                            # :538
        last = coord_predictions[-1] if iters > 0 else start
        coord_predictions2 = [start, start] + coord_predictions + [last, last]          # :474-475, :562-563
        return coord_predictions, coord_predictions2, vis_e, ffeat, ce
