#!/usr/bin/env python
"""Supervised evaluation calls (``Pips.forward`` with ``trajs_g``, ``no_grad``, ``is_train=False``): the torch path
against the CUDA path (``supervised='cuda'``) and plain inference, at the three shapes the reference's own scripts use.

    python tools/bench_supervised.py [--steps 3] [--warmup 1] [--only validation,flt,crohd] [--out FILE]

  validation  train.py:377-378   B=16 (4 clips x 2 x 2 flips), 384x512, N=768, stride 8, iters 4
  flt         test_on_flt.py:87  B=1, 384x512, N=16, stride 4, iters 6
  crohd       test_on_crohd.py   B=1, 768x1280, N=16, stride 4, iters 6

Per shape: the time of one call on each arm (the three arms alternate, every arm warmed up first, device-synchronised
host clock around each call), the peak of torch.cuda.max_memory_allocated over the first call of a fresh model on each
arm, the three losses of both supervised arms and their relative differences, and the score-loss kernel alone
(CUDA events over repeated launches on the pyramid and targets of the shape) against its MMA-issue and MUFU bounds.
Weights are seeded random (oracle.init_state_dict); inputs are seeded synthetic clips.  Prints one JSON document.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import ClockSampler  # noqa: E402
from oracle import pips_oracle as po  # noqa: E402
from pips_b200 import Pips, _lib as L  # noqa: E402
from pips_b200.supervised import score_targets  # noqa: E402

SHAPES = {
    "validation": dict(B=16, H=384, W=512, N=768, stride=8, iters=4),
    "flt": dict(B=1, H=384, W=512, N=16, stride=4, iters=6),
    "crohd": dict(B=1, H=768, W=1280, N=16, stride=4, iters=6),
}
DEV = "cuda:0"
MMA_FLOP_PER_CLK_SM = 8192          # dense bf16 tcgen05 rate per SM per clock (2250 TFLOP/s at 148 SMs, ~1.86 GHz)
MUFU_PER_CLK_SM = 16


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except Exception as e:                                 # noqa: BLE001
        return {"error": repr(e)}


def inputs(c, seed=0):
    B, H, W, N, stride = c["B"], c["H"], c["W"], c["N"], c["stride"]
    rgbs = po.smooth_video(B, 8, H, W, seed=seed + 1).to(DEV)
    xys = po.random_queries(B, N, H, W, seed=seed + 2).to(DEV)
    g = torch.Generator().manual_seed(seed + 3)
    tg = (xys.cpu()[:, None] + torch.cumsum(torch.randn(B, 8, N, 2, generator=g) * 2, 1)).to(DEV)
    vg = (torch.rand(B, 8, N, generator=g) > 0.2).float().to(DEV)
    va = (torch.rand(B, 8, N, generator=g) > 0.05).float().to(DEV)
    return rgbs, xys, tg, vg, va


def model(c, supervised):
    m = Pips(S=8, stride=c["stride"], supervised=supervised).to(DEV).eval()
    m.load_state_dict(po.init_state_dict(seed=0, head_scale=0.05), strict=True)
    return m


def arms(c, data):
    rgbs, xys, tg, vg, va = data
    sup = dict(trajs_g=tg, vis_g=vg, valids=va)
    return {"torch": lambda m: m(xys, rgbs, iters=c["iters"], **sup),
            "cuda": lambda m: m(xys, rgbs, iters=c["iters"], **sup),
            "plain": lambda m: m(xys, rgbs, iters=c["iters"])}


def peak_memory(c, data):
    out = {}
    for arm, fn in arms(c, data).items():
        m = model(c, "torch" if arm == "torch" else "cuda")
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        with torch.no_grad():
            fn(m)
        torch.cuda.synchronize()
        out[arm] = torch.cuda.max_memory_allocated() - base
        del m
        torch.cuda.empty_cache()
    return out


def score_kernel(c, m, data, reps=20):
    """pips_score_loss alone on the pyramid of an eager run of this shape: ms per launch and rates."""
    lib = L.load()
    rgbs, xys, tg, vg, va = data
    m.engine.use_graph = False
    with torch.no_grad():
        m(xys, rgbs, iters=1)                                    # leaves this shape's pyramid in the engine
    m.engine.use_graph = True
    pyr = m.engine._pyr
    B, N, iters = c["B"], c["N"], c["iters"]
    H8, W8 = c["H"] // c["stride"], c["W"] // c["stride"]
    ppad = -(-H8 * W8 // L.SCORE_TILE) * L.SCORE_TILE
    st = torch.cuda.current_stream().cuda_stream
    grid = torch.empty(2, B * 8, ppad, 128, dtype=torch.bfloat16, device=DEV)
    L.check(lib.pips_score_grid(pyr.f32_ptrs, B * 8, H8, W8, L.ptr(grid), st))
    target = score_targets(tg, vg, va, c["stride"], H8, W8)
    ffeats = torch.randn(B * N, 8, 128, device=DEV)
    partial = torch.empty(lib.pips_score_loss_scratch_floats(B * 8 * N, iters, H8, W8), device=DEV)

    def launch(it):
        L.check(lib.pips_score_loss(L.ptr(grid), B, 8, N, H8, W8, L.ptr(ffeats), L.ptr(target), 0, N, it, iters,
                                    L.ptr(partial), st))

    for it in range(iters):
        launch(it)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for r in range(reps):
        launch(r % iters)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(reps):
        L.check(lib.pips_score_grid(pyr.f32_ptrs, B * 8, H8, W8, L.ptr(grid), st))
    g1.record()
    torch.cuda.synchronize()
    try:
        hz = float(card()["clocks.sm"].split()[0]) * 1e6            # the SM clock right after the timed launches
    except (KeyError, ValueError, IndexError):
        hz = float("nan")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    elems = B * 8 * N * H8 * W8                                   # useful pixel-elements (score map entries)
    issued = B * 8 * (-(-N // 128) * 128) * ppad                  # what the MMA computes (M, N padded to tiles)
    mma_s = issued * 128 * 2 * 3 / (sms * MMA_FLOP_PER_CLK_SM * hz)
    mufu_s = issued * 2 / (sms * MUFU_PER_CLK_SM * hz)           # every row of an active warp runs ex2 + lg2
    return {"score_loss_ms": ms, "score_grid_ms": g0.elapsed_time(g1) / reps, "pixel_elements": elems,
            "pixel_elements_per_s": elems / (ms * 1e-3), "clock_hz_for_bounds": hz,
            "mma_issue_bound_ms": mma_s * 1e3, "mufu_bound_ms": mufu_s * 1e3,
            "bound_over_measured": max(mma_s, mufu_s) * 1e3 / ms}


def run_shape(name, c, steps, warmup):
    data = inputs(c)
    res = {"shape": c, "peak_bytes": peak_memory(c, data)}
    m = model(c, "cuda")
    fns = arms(c, data)
    times = {k: [] for k in fns}
    losses = {}
    with torch.no_grad():
        for arm, fn in fns.items():
            m.supervised = "torch" if arm == "torch" else "cuda"
            for _ in range(warmup):
                out = fn(m)
            if arm != "plain":
                losses[arm] = [float(x) for x in out[3]]
        sampler = ClockSampler(torch.device(DEV))
        sampler.start()
        for _ in range(steps):
            for arm, fn in fns.items():                          # alternate the arms
                m.supervised = "torch" if arm == "torch" else "cuda"
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(m)
                torch.cuda.synchronize()
                times[arm].append((time.perf_counter() - t0) * 1e3)
        res["clocks"] = sampler.stop()
    res["ms"] = {k: {"median": statistics.median(v), "min": min(v), "all": v} for k, v in times.items()}
    res["cuda_over_plain"] = res["ms"]["cuda"]["median"] / res["ms"]["plain"]["median"]
    res["torch_over_cuda"] = res["ms"]["torch"]["median"] / res["ms"]["cuda"]["median"]
    res["peak_torch_over_cuda"] = res["peak_bytes"]["torch"] / res["peak_bytes"]["cuda"]
    res["losses"] = losses
    res["losses_rel_diff"] = [abs(a - b) / max(abs(b), 1e-30) for a, b in zip(losses["cuda"], losses["torch"])]
    res["kernel"] = score_kernel(c, m, data)
    del m
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--only", default=",".join(SHAPES))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_supervised.py needs a CUDA device")
    doc = {"card": card(), "shapes": {}}
    for name in a.only.split(","):
        doc["shapes"][name] = run_shape(name, SHAPES[name], a.steps, a.warmup)
        print(name, json.dumps({k: doc["shapes"][name][k] for k in ("cuda_over_plain", "torch_over_cuda", "losses_rel_diff")}),
              file=sys.stderr, flush=True)
    text = json.dumps(doc, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
