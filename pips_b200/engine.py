"""Host driver of the CUDA refinement loop: weight packing, persistent buffers, launches.

Everything numerical happens in libpips_b200.so (include/pips_b200.h); torch is used for device
memory and streams only.  The driver mirrors the state machine of ``Pips.forward`` in the reference
(nets/pips.py:450-559): coords / ffeats state, one ``pips_refine_iter`` per iteration, vis head.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional

import torch

from . import _lib as L

S_FRAMES = 8
LATENT = 128

# PIPS_B200_NVTX=1: NVTX ranges around the phases of a forward (encoder, pyramid + initial features, every refinement
# iteration, visibility head) for `ncu --nvtx --nvtx-include "pips/iter3/"` and timeline tools (SURVEY.md section 5).
_NVTX = os.environ.get("PIPS_B200_NVTX", "0") == "1"


class nvtx_range:
    def __init__(self, name: str):
        self.name = name

    def __enter__(self):
        if _NVTX:
            torch.cuda.nvtx.range_push(self.name)

    def __exit__(self, *exc):
        if _NVTX:
            torch.cuda.nvtx.range_pop()
        return False


def _round_up(v: int, m: int) -> int:
    return (v + m - 1) // m * m


class PackedWeights:
    """Kernel-layout copies of the DeltaBlock / head parameters.

    Dense-layer weights are kept as nn.Linear stores them ((out, in) == N x K, K-major), split into a
    bf16 (hi, lo) pair for the tcgen05 path; the first Linear's K is zero-padded 519 -> 576 and the
    last Linear's N 1040 -> 1280 so that TMA boxes never leave the allocation.

    ``self.t`` holds every tensor under a stable name ("layer3.fc1_w_hi", "head_b", ...); the names are
    the fields of ``pips_weights`` / ``pips_layer_weights`` in include/pips_b200.h, which is also the
    manifest of the on-disk pack (pips_b200/pack.py, SURVEY.md section 8f-4).
    """

    def __init__(self, module=None, stream=None, tensors: Optional[Dict[str, torch.Tensor]] = None):
        self.c = L.Weights()
        if tensors is not None:
            self.t = dict(tensors)
            self.device = self.t["gn_w"].device
        else:
            self.t = self._pack(module, stream)
            self.device = self.t["gn_w"].device
        if self.device.type != "cuda":
            raise L.PipsCudaError("pips_b200: the refinement path needs the module on a CUDA device")
        self._bind()

    @staticmethod
    def _pack(module, stream) -> Dict[str, torch.Tensor]:
        lib = L.load()
        sd = {k: v.detach() for k, v in module.state_dict().items()}
        dev = sd["norm.weight"].device
        if dev.type != "cuda":
            raise L.PipsCudaError("pips_b200: the refinement path needs the module on a CUDA device")
        t: Dict[str, torch.Tensor] = {}

        def f32(name, v):
            t[name] = v.to(torch.float32).contiguous().clone()

        def split(name, v):
            f32(name + "_f32", v)
            src = t[name + "_f32"]
            hi = torch.empty(src.shape, dtype=torch.bfloat16, device=dev)
            lo = torch.empty(src.shape, dtype=torch.bfloat16, device=dev)
            L.check(lib.pips_split_bf16(L.ptr(src), L.ptr(hi), L.ptr(lo), src.numel(), stream), "pips_split_bf16")
            t[name + "_hi"], t[name + "_lo"] = hi, lo

        td = "delta_block.to_delta"
        w0 = torch.zeros(L.DIM, L.KPAD, dtype=torch.float32, device=dev)
        w0[:, :519] = sd[f"{td}.0.weight"]
        split("in_w", w0)
        f32("in_b", sd[f"{td}.0.bias"])
        for l in range(L.DEPTH):
            p, q = f"{td}.{l + 1}", f"layer{l}."
            f32(q + "ln1_w", sd[p + ".0.norm.weight"])
            f32(q + "ln1_b", sd[p + ".0.norm.bias"])
            f32(q + "tok_w1", sd[p + ".0.fn.0.weight"].reshape(4 * S_FRAMES, S_FRAMES))
            f32(q + "tok_b1", sd[p + ".0.fn.0.bias"])
            f32(q + "tok_w2", sd[p + ".0.fn.3.weight"].reshape(S_FRAMES, 4 * S_FRAMES))
            f32(q + "tok_b2", sd[p + ".0.fn.3.bias"])
            f32(q + "ln2_w", sd[p + ".1.norm.weight"])
            f32(q + "ln2_b", sd[p + ".1.norm.bias"])
            split(q + "fc1_w", sd[p + ".1.fn.0.weight"])
            f32(q + "fc1_b", sd[p + ".1.fn.0.bias"])
            split(q + "fc2_w", sd[p + ".1.fn.3.weight"])
            f32(q + "fc2_b", sd[p + ".1.fn.3.bias"])
        f32("out_ln_w", sd[f"{td}.13.weight"])
        f32("out_ln_b", sd[f"{td}.13.bias"])
        wh = torch.zeros(L.HEAD_PAD, L.DIM, dtype=torch.float32, device=dev)
        wh[:L.HEAD] = sd[f"{td}.15.weight"]
        split("head_w", wh)
        f32("head_b", sd[f"{td}.15.bias"])
        f32("gn_w", sd["norm.weight"])
        f32("gn_b", sd["norm.bias"])
        f32("upd_w", sd["ffeat_updater.0.weight"])
        f32("upd_b", sd["ffeat_updater.0.bias"])
        f32("vis_w", sd["vis_predictor.0.weight"].reshape(-1))
        f32("vis_b", sd["vis_predictor.0.bias"])
        return t

    LAYER_FIELDS = ("ln1_w", "ln1_b", "tok_w1", "tok_b1", "tok_w2", "tok_b2", "ln2_w", "ln2_b",
                    "fc1_w_hi", "fc1_w_lo", "fc1_w_f32", "fc1_b", "fc2_w_hi", "fc2_w_lo", "fc2_w_f32", "fc2_b")
    TOP_FIELDS = ("in_w_hi", "in_w_lo", "in_w_f32", "in_b", "out_ln_w", "out_ln_b", "head_w_hi", "head_w_lo",
                  "head_w_f32", "head_b", "gn_w", "gn_b", "upd_w", "upd_b", "vis_w", "vis_b")

    @classmethod
    def names(cls):
        return list(cls.TOP_FIELDS) + [f"layer{l}.{f}" for l in range(L.DEPTH) for f in cls.LAYER_FIELDS]

    def _bind(self) -> None:
        """Point the C struct at the named tensors (which must stay alive as long as ``self``)."""
        missing = [n for n in self.names() if n not in self.t]
        if missing:
            raise L.PipsCudaError(f"pips_b200: weight pack lacks {missing[:4]}{' ...' if len(missing) > 4 else ''}")
        for n in self.names():
            v = self.t[n]
            if v.device != self.device or not v.is_contiguous():
                raise L.PipsCudaError(f"pips_b200: weight pack tensor {n} is not a contiguous tensor on {self.device}")
        for f in self.TOP_FIELDS:
            setattr(self.c, f, L.ptr(self.t[f]))
        for l in range(L.DEPTH):
            for f in self.LAYER_FIELDS:
                setattr(self.c.layer[l], f, L.ptr(self.t[f"layer{l}.{f}"]))


class Workspace:
    """Mixer activations for up to ``seqs`` particle tracks ((b, n) pairs)."""

    def __init__(self, seqs: int, precision: int, device):
        self.seqs = seqs
        rows = _round_up(seqs * S_FRAMES, 256)        # whole 256-row CTA-pair tiles
        sq = _round_up(seqs, 256)
        self.c = L.Workspace()
        self.c.rows_alloc, self.c.seqs_alloc = rows, sq
        self.keep: Dict[str, torch.Tensor] = {}

        def alloc(name, r, c, dtype):
            t = torch.zeros(r, c, dtype=dtype, device=device)
            self.keep[name] = t
            setattr(self.c, name, L.ptr(t))

        alloc("x", rows, L.DIM, torch.float32)
        alloc("delta", sq, L.HEAD, torch.float32)
        if precision == L.PREC_F32:
            alloc("x0_f32", rows, L.KPAD, torch.float32)
            alloc("y_f32", rows, L.DIM, torch.float32)
            alloc("h_f32", rows, L.HIDDEN, torch.float32)
            alloc("p_f32", sq, L.DIM, torch.float32)
        else:
            parts = ("hi", "lo") if precision == L.PREC_BF16X3 else ("hi",)
            for part in parts:
                alloc(f"x0_{part}", rows, L.KPAD, torch.bfloat16)
                alloc(f"y_{part}", rows, L.DIM, torch.bfloat16)
                alloc(f"h_{part}", rows, L.HIDDEN, torch.bfloat16)
                alloc(f"p_{part}", sq, L.DIM, torch.bfloat16)


class Pyramid:
    """4-level channels-last correlation pyramid (nets/pips.py:346-352)."""

    def __init__(self, frames: int, H: int, W: int, feat_dtype: int, device):
        self.frames, self.H, self.W, self.feat_dtype = frames, H, W, feat_dtype
        self.f32, self.bf16 = [], []
        h, w = H, W
        for _ in range(L.LEVELS):
            self.f32.append(torch.empty(frames, h, w, LATENT, dtype=torch.float32, device=device))
            if feat_dtype == L.FEAT_BF16:
                self.bf16.append(torch.empty(frames, h, w, LATENT, dtype=torch.bfloat16, device=device))
            h, w = h // 2, w // 2
        self.f32_ptrs = L.ptr_array(self.f32)
        self.bf16_ptrs = L.ptr_array(self.bf16) if self.bf16 else None

    def levels(self):
        return self.bf16 if self.feat_dtype == L.FEAT_BF16 else self.f32

    def build(self, fmaps: torch.Tensor, stream) -> None:
        """fmaps: (frames,128,H,W) fp32, either NCHW-contiguous or channels-last (NHWC memory)."""
        lib = L.load()
        assert fmaps.dtype == torch.float32
        if fmaps.is_contiguous():
            L.check(lib.pips_pyramid_build(L.ptr(fmaps), self.frames, self.H, self.W, self.f32_ptrs,
                                           self.bf16_ptrs, stream), "pips_pyramid_build")
        else:
            assert fmaps.permute(0, 2, 3, 1).is_contiguous(), "fmaps must be NCHW- or NHWC-contiguous"
            L.check(lib.pips_pyramid_build_nhwc(L.ptr(fmaps), self.frames, self.H, self.W, self.f32_ptrs,
                                                self.bf16_ptrs, stream), "pips_pyramid_build_nhwc")


class RefineEngine:
    """Runs the refinement loop for one model on one device."""

    def __init__(self, precision: str = "bf16x3", feat_dtype: str = "fp32", max_seqs: int = 32768):
        if precision not in L.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(L.PRECISIONS)}")
        if feat_dtype not in L.FEAT_DTYPES:
            raise ValueError(f"feat_dtype must be one of {sorted(L.FEAT_DTYPES)}")
        self.precision = L.PRECISIONS[precision]
        self.feat_dtype = L.FEAT_DTYPES[feat_dtype]
        self.max_seqs = max_seqs
        self._weights: Optional[PackedWeights] = None
        self._weights_key = None
        self._ws: Optional[Workspace] = None
        self._pyr: Optional[Pyramid] = None
        self._times = None
        self._plans: Dict[tuple, "_GraphPlan"] = {}
        self.use_graph = os.environ.get("PIPS_B200_GRAPH", "1") != "0"
        self.launches = 0                       # kernels launched by the last refine() call

    # ------------------------------------------------------------------ caches
    @staticmethod
    def _stream() -> int:
        return torch.cuda.current_stream().cuda_stream

    def weights(self, module) -> PackedWeights:
        key = tuple((p.data_ptr(), p._version) for p in module.parameters())
        if self._weights is None or key != self._weights_key:
            self._plans.clear()                                   # captured graphs point into the old pack
            self._weights = PackedWeights(module, self._stream())
            self._weights_key = key
        return self._weights

    def invalidate(self, graphs_only: bool = False) -> None:
        """Drop the captured CUDA graphs (and, unless ``graphs_only``, the packed weights).  The caches are keyed by
        (data_ptr, _version) of every parameter, which in-place edits through ``.data`` (a manual EMA,
        ``p.data.copy_()``) do not change: call this after such an edit.  Also used when the buffers a captured
        graph points into go away (peer slabs re-allocated)."""
        self._plans.clear()
        if not graphs_only:
            self._weights, self._weights_key = None, None

    def adopt_weights(self, module, packed: PackedWeights) -> None:
        """Use an already packed weight set (pips_b200/pack.py) for ``module``'s current parameters."""
        self._plans.clear()
        self._weights = packed
        self._weights_key = tuple((p.data_ptr(), p._version) for p in module.parameters())

    def workspace(self, seqs: int, device) -> Workspace:
        if self._ws is None or self._ws.seqs < seqs or next(iter(self._ws.keep.values())).device != device:
            self._ws = None
            self._ws = Workspace(seqs, self.precision, device)
        return self._ws

    def pyramid(self, frames: int, H: int, W: int, device) -> Pyramid:
        p = self._pyr
        if p is None or (p.frames, p.H, p.W) != (frames, H, W) or p.f32[0].device != device:
            self._pyr = None
            self._pyr = Pyramid(frames, H, W, self.feat_dtype, device)
        return self._pyr

    def times(self, device) -> torch.Tensor:
        if self._times is None or self._times.device != device:
            # computed on the host exactly as the reference does (nets/pips.py:519); the sin/cos
            # embedding multiplies it by up to 968.75, so the fp32 bit pattern matters
            self._times = torch.linspace(0, S_FRAMES, S_FRAMES, dtype=torch.float32).to(device)
        return self._times

    # ------------------------------------------------------------------ the loop
    def _enqueue(self, lib, wc, pyr: Pyramid, ws: Workspace, fmaps2d, c, c0, ffeat, ffeats, feat_init, out, vis,
                 B, S, nc, H8, W8, iters, stride, on_iter=None, build_pyramid=True, frame_base=None, T=0,
                 heat=None, score_loss=None, peer=None, peer_n0=0) -> int:
        """Enqueue every launch of one forward for ``nc`` particles on the current stream: pyramid, initial
        features, ``iters`` refinement iterations, visibility head.  Returns the number of kernels launched.
        ``score_loss`` (``_ScoreLoss``): also the score-map loss of these particles (nets/pips.py:58-90)."""
        st = self._stream()
        launches = 0
        if build_pyramid:
            with nvtx_range("pips/pyramid"):
                pyr.build(fmaps2d, st)
            launches += 4
            if score_loss is not None:
                L.check(lib.pips_score_grid(pyr.f32_ptrs, B * S, H8, W8, L.ptr(score_loss.grid), st), "pips_score_grid")
                launches += 1
        c0.copy_(c)
        if feat_init is None:
            L.check(lib.pips_init_gather(L.ptr(pyr.f32[0]), B, S, nc, H8, W8, L.ptr(c), L.ptr(frame_base), T, L.ptr(ffeat),
                                         L.ptr(ffeats), st), "pips_init_gather")
            launches += 1
        else:
            ffeat.copy_(feat_init.reshape(B * nc, LATENT))
            ffeats.copy_(ffeat.unsqueeze(1).expand(-1, S, -1))
        lvl = pyr.levels()
        prob = L.Problem()
        prob.B, prob.S, prob.N, prob.H, prob.W = B, S, nc, H8, W8
        prob.feat_dtype, prob.precision = self.feat_dtype, self.precision
        for i in range(L.LEVELS):
            prob.lvl[i] = L.ptr(lvl[i])
        prob.times, prob.coords, prob.coords0, prob.ffeats = L.ptr(self.times(c.device)), L.ptr(c), L.ptr(c0), L.ptr(ffeats)
        prob.stride = float(stride)
        prob.frame_base, prob.frames_per_batch = L.ptr(frame_base), T
        if heat is not None:
            sel, slot, fcps = heat                  # local particle indices, output slots, (B,S,I,n_sel_total,H8,W8)
            scratch = torch.empty(lib.pips_heatmap_scratch_floats(B * S, sel.numel(), H8, W8), dtype=torch.float32,
                                  device=c.device)
            lvl_ptrs = L.ptr_array(lvl)
        if peer is not None:                        # particle-sharded: predictions go straight into every rank's slab
            prob.peer.n_peers, prob.peer.n_total = peer.slab.world, peer.n_total
            prob.peer.n_offset = peer.n_offset + peer_n0
        for it in range(iters):
            if peer is not None:
                for r, a in enumerate(peer.coord_bases(it)):
                    prob.peer.out[r] = a
            if heat is not None:                    # nets/pips.py:502-511: score map of the state the iteration starts from
                L.check(lib.pips_heatmap(lvl_ptrs, self.feat_dtype, B, S, nc, H8, W8, L.ptr(ffeats), L.ptr(sel), L.ptr(slot),
                                         sel.numel(), L.ptr(scratch), L.ptr(fcps[0, 0, it]),
                                         fcps.stride(1), st), "pips_heatmap")
                launches += 1 + (sel.numel() + 31) // 32
            if score_loss is not None:              # nets/pips.py:502-511 + :58-90: loss terms of the starting state
                sl = score_loss
                L.check(lib.pips_score_loss(L.ptr(sl.grid), B, S, nc, H8, W8, L.ptr(ffeats), L.ptr(sl.target), peer_n0,
                                            sl.n_total, it, iters, L.ptr(sl.partial), st), "pips_score_loss")
                launches += 1
            with nvtx_range(f"pips/iter{it}"):
                L.check(lib.pips_refine_iter(C.byref(prob), C.byref(wc), C.byref(ws.c), L.ptr(out[it]), st), "pips_refine_iter")
            launches += 1 + (1 + 3 * L.DEPTH + 2) + 1
            if on_iter is not None:
                on_iter(it, out[it])
        with nvtx_range("pips/vis_head"):
            L.check(lib.pips_vis_head(L.ptr(ffeats), wc.vis_w, wc.vis_b, L.ptr(vis), B, S, nc, st), "pips_vis_head")
        if score_loss is not None and peer_n0 + nc == score_loss.n_total:      # the last chunk: reduce all partials
            L.check(lib.pips_score_loss_finalize(L.ptr(score_loss.target), score_loss.target.numel(), iters, H8, W8,
                                                 L.ptr(score_loss.partial), L.ptr(score_loss.ce), st), "pips_score_loss_finalize")
            launches += 2
        return launches + 1

    def refine(self, module, fmaps: torch.Tensor, coords: torch.Tensor, feat_init: Optional[torch.Tensor],
               iters: int, stride: float, on_iter=None, frame_base: Optional[torch.Tensor] = None,
               reuse_pyramid: bool = False, heat_sel: Optional[torch.Tensor] = None,
               heat_out: Optional[torch.Tensor] = None, peer=None, score_target: Optional[torch.Tensor] = None):
        """fmaps (B,S,128,H8,W8) fp32, coords (B,S,N,2) fp32 in feature-map pixels.
        Returns preds (iters,B,S,N,2) in input pixels, vis_e (B,S,N) logits, ffeat (B,N,128).
        ``on_iter(it, coords_px)`` (optional) is called once per iteration when the particles fit one
        chunk -- the sharded path hangs its per-iteration all-gather there.
        ``frame_base`` (B,N) int32 (optional): chained tracking -- fmaps then holds T >= 1 frames per batch
        element and track (b,n) works on frames min(frame_base[b,n] + s, T-1), s = 0..7.
        ``reuse_pyramid``: the pyramid built by the previous call is still valid (same fmaps; chained rounds).
        ``heat_sel`` (n_sel,) particle indices + ``heat_out`` (B,S,iters,n_sel,H8,W8) fp32: also write the score maps
        of those particles (nets/pips.py:504-511) at the start of every iteration (eager launches, no graph).
        ``peer`` (pips_b200.peer.PeerPlan): this call refines one rank's slice of a particle-sharded run; the update
        kernel also stores every iteration's prediction into all ranks' slabs (the caller runs the barriers).
        ``score_target`` (B,S,N) int32 (pips_b200.supervised.score_targets): also compute the score-map loss
        (nets/pips.py:58-90) of the run; the result is then (preds, vis_e, ffeat, ce) with ce a 0-dim fp32 tensor.  The
        score maps are never stored, and preds / vis_e / ffeat are those of the same call without it."""
        lib = L.load()
        B, T, Cc, H8, W8 = fmaps.shape
        S = coords.shape[1]
        if S != S_FRAMES or Cc != LATENT or (frame_base is None and T != S):
            raise L.PipsCudaError(f"pips_b200 CUDA path supports S=8, C=128 (got S={S}, T={T}, C={Cc})")
        if frame_base is not None:
            frame_base = frame_base.to(device=fmaps.device, dtype=torch.int32).contiguous()
        N = coords.shape[2]
        dev = fmaps.device
        w = self.weights(module)
        fmaps2d = fmaps.reshape(B * T, Cc, H8, W8)                  # a view for both NCHW and channels-last inputs
        if not fmaps2d.is_contiguous() and not fmaps2d.permute(0, 2, 3, 1).is_contiguous():
            fmaps2d = fmaps2d.contiguous()
        chunk = max(1, self.max_seqs // B)

        if heat_sel is not None:
            if frame_base is not None:
                raise L.PipsCudaError("pips_b200: score maps are not defined for chained windows")
            heat_sel = heat_sel.to(device=dev, dtype=torch.int32).contiguous()
            n_sel = heat_sel.numel()
            assert n_sel > 0 and int(heat_sel.min()) >= 0 and int(heat_sel.max()) < N, "heat_sel out of range"
            assert heat_out is not None and tuple(heat_out.shape) == (B, S, iters, n_sel, H8, W8) \
                and heat_out.dtype == torch.float32 and heat_out.is_contiguous() and heat_out.device == dev
        score = score_target is not None
        if score:
            if frame_base is not None or heat_sel is not None or peer is not None or iters <= 0:
                raise L.PipsCudaError("pips_b200: the score-map loss needs iters > 0 and a plain, unsharded forward")
            assert tuple(score_target.shape) == (B, S, N) and score_target.dtype == torch.int32 \
                and score_target.device == dev, "score_target must be (B,S,N) int32 on the device of fmaps"
        if N <= chunk and self.use_graph and iters > 0 and frame_base is None and heat_sel is None:
            plan = self._plan(w, B, S, N, H8, W8, iters, float(stride), feat_init is not None, dev,
                              nhwc=not fmaps2d.is_contiguous(), peer=peer, score=score)
            preds, vis, ffeat, ce = plan.run(fmaps2d, coords, feat_init, score_target)
            self.launches = plan.launches
            if on_iter is not None:
                for it in range(iters):
                    on_iter(it, preds[it])
            return (preds, vis, ffeat, ce) if score else (preds, vis, ffeat)

        pyr = self.pyramid(B * T, H8, W8, dev)
        preds = torch.empty(iters, B, S, N, 2, dtype=torch.float32, device=dev)
        vis = torch.empty(B, S, N, dtype=torch.float32, device=dev)
        ffeat_out = torch.empty(B, N, LATENT, dtype=torch.float32, device=dev)
        sl = _ScoreLoss(B, S, N, H8, W8, iters, dev, score_target.contiguous()) if score else None
        self.launches = 0
        for n0 in range(0, N, chunk):
            n1 = min(N, n0 + chunk)
            nc = n1 - n0
            whole = nc == N
            c = (coords if whole else coords[:, :, n0:n1]).contiguous().clone()
            c0 = torch.empty_like(c)
            ffeat = torch.empty(B * nc, LATENT, dtype=torch.float32, device=dev)
            ffeats = torch.empty(B * nc, S, LATENT, dtype=torch.float32, device=dev)
            fi = None if feat_init is None else (feat_init if whole else feat_init[:, n0:n1])
            ws = self.workspace(B * nc, dev)
            out = preds if whole else torch.empty(iters, B, S, nc, 2, dtype=torch.float32, device=dev)
            v = vis if whole else torch.empty(B, S, nc, dtype=torch.float32, device=dev)
            fb = None if frame_base is None else (frame_base if whole else frame_base[:, n0:n1].contiguous())
            heat = None
            if heat_sel is not None:
                inside = ((heat_sel >= n0) & (heat_sel < n1)).nonzero().flatten()
                if inside.numel() > 0:
                    heat = ((heat_sel[inside] - n0).to(torch.int32).contiguous(), inside.to(torch.int32).contiguous(), heat_out)
            self.launches += self._enqueue(lib, w.c, pyr, ws, fmaps2d, c, c0, ffeat, ffeats, fi, out, v, B, S, nc, H8, W8,
                                           iters, stride, on_iter if whole else None,
                                           build_pyramid=(n0 == 0 and not reuse_pyramid), frame_base=fb, T=T, heat=heat,
                                           score_loss=sl, peer=peer, peer_n0=n0)
            if not whole:
                preds[:, :, :, n0:n1] = out
                vis[:, :, n0:n1] = v
            ffeat_out[:, n0:n1] = ffeat.reshape(B, nc, LATENT)
        if score:
            return preds, vis, ffeat_out, sl.ce.reshape(())
        return preds, vis, ffeat_out

    def _plan(self, w: PackedWeights, B, S, N, H8, W8, iters, stride, has_feat, dev, nhwc=False, peer=None,
              score=False) -> "_GraphPlan":
        key = (id(w), B, S, N, H8, W8, iters, stride, has_feat, str(dev), nhwc, None if peer is None else peer.key, score)
        plan = self._plans.get(key)
        if plan is None:
            while len(self._plans) >= 2:                          # each plan owns a full workspace
                self._plans.pop(next(iter(self._plans)))
            plan = _GraphPlan(self, w, B, S, N, H8, W8, iters, stride, has_feat, dev, nhwc, peer, score)
            self._plans[key] = plan
        else:
            self._plans[key] = self._plans.pop(key)               # LRU order
        return plan

    # ------------------------------------------------------------------ instrumentation
    def profile_iteration(self, module, fmaps: torch.Tensor, coords: torch.Tensor, stride: float, reps: int = 3):
        """Re-runs one refinement iteration kernel by kernel (the same launches pips_refine_iter makes,
        same buffers, back to back) with CUDA events around every launch.  Returns
        {kernel class: [ms, ...]} -- the source of the live roofline numbers in bench.py."""
        lib = L.load()
        B, S, Cc, H8, W8 = fmaps.shape
        N = coords.shape[2]
        if B * N > self.max_seqs:
            N = self.max_seqs // B
            coords = coords[:, :, :N]
        dev = fmaps.device
        st = self._stream()
        w = self.weights(module).c
        pyr = self.pyramid(B * S, H8, W8, dev)
        pyr.build(fmaps.reshape(B * S, Cc, H8, W8).contiguous(), st)
        lvl = L.ptr_array(pyr.levels())
        c = coords.contiguous().clone()
        c0 = c.clone()
        ffeat = torch.empty(B * N, LATENT, dtype=torch.float32, device=dev)
        ffeats = torch.empty(B * N, S, LATENT, dtype=torch.float32, device=dev)
        L.check(lib.pips_init_gather(L.ptr(pyr.f32[0]), B, S, N, H8, W8, L.ptr(c), None, 0, L.ptr(ffeat), L.ptr(ffeats), st))
        ws = self.workspace(B * N, dev).c
        times = self.times(dev)
        out = torch.empty(B, S, N, 2, dtype=torch.float32, device=dev)
        seqs, M = B * N, B * N * S
        f32, x3 = self.precision == L.PREC_F32, self.precision == L.PREC_BF16X3
        rec: Dict[str, list] = {}

        def timed(name, fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            L.check(fn(), name)
            e1.record()
            rec.setdefault(name, []).append((e0, e1))

        def dense(name, a, lda, a_rows, wt, ldw, w_rows, Mv, Nv, Kv, bias, epi, o32, ldo, oh, ldh):
            if f32:
                o = oh[2] if epi == L.EPI_BIAS_GELU else o32
                ld = ldh if epi == L.EPI_BIAS_GELU else ldo
                timed(name, lambda: lib.pips_gemm_f32(a[2], lda, wt[2], ldw, Mv, Nv, Kv, bias, epi, o, ld, st))
            else:
                timed(name, lambda: lib.pips_gemm_tc(a[0], a[1] if x3 else None, lda, a_rows, wt[0], wt[1] if x3 else None, ldw,
                                                     w_rows, Mv, Nv, Kv, bias, epi, o32, ldo, oh[0], oh[1] if x3 else None, ldh, st))

        for _ in range(reps):
            timed("corr_gather", lambda: lib.pips_corr_gather(
                lvl, self.feat_dtype, B, S, N, H8, W8, L.ptr(c), L.ptr(ffeats), L.ptr(times), None, 0,
                None if f32 else ws.x0_hi, ws.x0_lo if x3 else None, ws.x0_f32 if f32 else None, L.KPAD, st))
            dense("gemm_in", (ws.x0_hi, ws.x0_lo, ws.x0_f32), L.KPAD, ws.rows_alloc, (w.in_w_hi, w.in_w_lo, w.in_w_f32), L.KPAD,
                  L.DIM, M, L.DIM, L.KPAD, w.in_b, L.EPI_BIAS, ws.x, L.DIM, (None, None, None), 0)
            for l in range(L.DEPTH):
                lw = w.layer[l]
                timed("tokenmix", lambda: lib.pips_tokenmix(
                    ws.x, seqs, lw.ln1_w, lw.ln1_b, lw.tok_w1, lw.tok_b1, lw.tok_w2, lw.tok_b2, lw.ln2_w, lw.ln2_b,
                    None if f32 else ws.y_hi, ws.y_lo if x3 else None, ws.y_f32 if f32 else None, st))
                dense("gemm_fc1", (ws.y_hi, ws.y_lo, ws.y_f32), L.DIM, ws.rows_alloc, (lw.fc1_w_hi, lw.fc1_w_lo, lw.fc1_w_f32),
                      L.DIM, L.HIDDEN, M, L.HIDDEN, L.DIM, lw.fc1_b, L.EPI_BIAS_GELU, None, 0, (ws.h_hi, ws.h_lo, ws.h_f32), L.HIDDEN)
                dense("gemm_fc2", (ws.h_hi, ws.h_lo, ws.h_f32), L.HIDDEN, ws.rows_alloc, (lw.fc2_w_hi, lw.fc2_w_lo, lw.fc2_w_f32),
                      L.HIDDEN, L.DIM, M, L.DIM, L.HIDDEN, lw.fc2_b, L.EPI_BIAS_RESID, ws.x, L.DIM, (None, None, None), 0)
            timed("ln_pool", lambda: lib.pips_ln_pool(ws.x, seqs, w.out_ln_w, w.out_ln_b, None if f32 else ws.p_hi,
                                                      ws.p_lo if x3 else None, ws.p_f32 if f32 else None, st))
            dense("gemm_head", (ws.p_hi, ws.p_lo, ws.p_f32), L.DIM, ws.seqs_alloc, (w.head_w_hi, w.head_w_lo, w.head_w_f32), L.DIM,
                  L.HEAD_PAD, seqs, L.HEAD, L.DIM, w.head_b, L.EPI_BIAS, ws.delta, L.HEAD, (None, None, None), 0)
            timed("update", lambda: lib.pips_update(ws.delta, L.ptr(c), L.ptr(c0), L.ptr(ffeats), w.gn_w, w.gn_b, w.upd_w, w.upd_b,
                                                    L.ptr(out), float(stride), B, S, N, st))
        torch.cuda.synchronize()
        return {k: [a.elapsed_time(b) for a, b in v] for k, v in rec.items()}, dict(B=B, S=S, N=N, M=M)


class _ScoreLoss:
    """Device buffers of the score-map loss of one forward: ``target`` (B,S,N) int32 (pixel index or -1), the bf16
    (hi, lo) grid ``Gr`` of pips_score_grid, the per-(track, pixel block) ``partial`` sums and the ``ce`` scalar."""

    def __init__(self, B, S, N, H8, W8, iters, dev, target=None):
        lib = L.load()
        ppad = _round_up(H8 * W8, L.SCORE_TILE)
        self.n_total = N
        self.target = target if target is not None else torch.full((B, S, N), -1, dtype=torch.int32, device=dev)
        self.grid = torch.empty(2, B * S, ppad, LATENT, dtype=torch.bfloat16, device=dev)
        self.partial = torch.empty(lib.pips_score_loss_scratch_floats(B * S * N, iters, H8, W8), dtype=torch.float32,
                                   device=dev)
        self.ce = torch.zeros(1, dtype=torch.float32, device=dev)


class _GraphPlan:
    """One captured CUDA graph of a whole forward (pyramid .. vis head) for a fixed problem signature,
    with its own static buffers; replayed with new inputs copied in.  ~250 launches per forward collapse
    into one graph launch, which is what matters for small problems (demo / chained windows)."""

    def __init__(self, eng: RefineEngine, w: PackedWeights, B, S, N, H8, W8, iters, stride, has_feat, dev, nhwc=False,
                 peer=None, score=False):
        lib = L.load()
        self.w = w
        self.peer = peer                              # the captured update kernels store into these slabs
        self.iters = iters
        self.pyr = Pyramid(B * S, H8, W8, eng.feat_dtype, dev)
        self.ws = Workspace(B * N, eng.precision, dev)
        f32 = dict(dtype=torch.float32, device=dev)
        self.fmaps_nchw = torch.zeros(B * S, LATENT, H8, W8, **f32)
        self.fmaps_nhwc = self.fmaps_nchw.view(B * S, H8, W8, LATENT).permute(0, 3, 1, 2)   # same storage, NHWC strides
        self.c = torch.zeros(B, S, N, 2, **f32)
        self.c0 = torch.zeros_like(self.c)
        self.feat_in = torch.zeros(B, N, LATENT, **f32) if has_feat else None
        self.ffeat = torch.zeros(B * N, LATENT, **f32)
        self.ffeats = torch.zeros(B * N, S, LATENT, **f32)
        self.preds = torch.zeros(iters, B, S, N, 2, **f32)
        self.vis = torch.zeros(B, S, N, **f32)
        self.shape = (B, N)
        self.score = _ScoreLoss(B, S, N, H8, W8, iters, dev) if score else None      # static target / partials / ce
        eng.times(dev)

        self.nhwc = nhwc

        def enqueue():
            return eng._enqueue(lib, w.c, self.pyr, self.ws, self.fmaps_nhwc if nhwc else self.fmaps_nchw, self.c, self.c0,
                                self.ffeat, self.ffeats, self.feat_in, self.preds, self.vis, B, S, N, H8, W8, iters, stride,
                                score_loss=self.score, peer=peer)

        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            self.launches = enqueue()                 # eager warm-up: function attributes, lazy module load
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            enqueue()

    def run(self, fmaps2d, coords, feat_init, score_target=None):
        B, N = self.shape
        (self.fmaps_nhwc if self.nhwc else self.fmaps_nchw).copy_(fmaps2d)
        self.c.copy_(coords)
        if self.feat_in is not None:
            self.feat_in.copy_(feat_init)
        if self.score is not None:
            self.score.target.copy_(score_target)
        self.graph.replay()
        ce = self.score.ce.reshape(()).clone() if self.score is not None else None
        return self.preds.clone(), self.vis.clone(), self.ffeat.reshape(B, N, LATENT).clone(), ce
