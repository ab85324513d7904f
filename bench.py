#!/usr/bin/env python
"""Benchmark of the PIPs refinement hot path (BASELINE.json metric: particle-frame updates/s).

    python bench.py --gpus 1 --steps 20 --warmup 5            # this repo's CUDA path on 1 GPU
    torchrun ... bench.py --gpus N ...                        # one rank per GPU, particle-sharded (weak scaling)
    python bench.py --impl reference ...                      # the reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR                    # also save the last timed step's outputs as .npy

A step is one ``Pips.forward(xys, rgbs, iters=6)`` over one synthetic batch:
  N=1   BASELINE configs[1]: B=4, S=8, 384x512, N=1024, iters=6, stride 8
  N>1   per-GPU work fixed (1024 particles per rank), global N = 1024*G (G=4 is configs[2], N=4096)
``value`` counts B*S*N_global*iters updates per second of the max-over-ranks device time with the
inputs resident in HBM; ``e2e`` runs the same call from pinned host buffers with the H2D / D2H copies
inside the timed region.  One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B, S, H, W, N_PER_GPU, ITERS, STRIDE = 4, 8, 384, 512, 1024, 6, 8
UNIT_FLOP = 51.78e6                       # mixer matmul FLOPs per particle-frame update (SURVEY.md 8d)
METRIC = "particle_frame_updates_per_sec"
UNIT = "updates/s"


def peaks():
    p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            m = json.load(f)
        p.update({k: float(m[k]) for k in ("hbm_gbs", "bf16_tflops", "bf16_tflops_sustained") if k in m})
        p["source"] = "measured"
    except Exception:
        pass
    return p


class ClockSampler:
    """SM clock and throttle reasons of THIS rank's GPU during the timed region, read through NVML (what nvidia-smi
    itself reads) from a thread of this process, every 100 ms.  A separate nvidia-smi process polling in a loop
    attaches to every GPU of the box and was the one thing the device-timed loop had that the e2e loop did not;
    the in-process query touches only this GPU.  Falls back to an nvidia-smi poller if NVML cannot be loaded."""
    REASONS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, device: torch.device):
        self.device, self.mhz, self.mask, self.max_mhz, self.stop_flag, self.thread, self.smi = device, [], 0, None, False, None, None
        self.index = device.index or 0

    def _handle(self, nv):
        try:
            uuid = str(torch.cuda.get_device_properties(self.device).uuid)
            return nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            return nv.nvmlDeviceGetHandleByIndex(self.index)

    def _poll(self, nv, h):
        while not self.stop_flag:
            try:
                self.mhz.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
            except Exception:
                pass
            time.sleep(0.1)

    def mark(self):
        """Forget the samples taken so far (warm-up): the record covers the timed region only."""
        self.mhz, self.mask = [], 0
        if self.smi is not None:
            self.lines = []

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = self._handle(nv)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, args=(nv, h), daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None
            self._start_smi()

    def _start_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.smi = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                                         str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.lines = []
            self.thread = threading.Thread(target=lambda: self.lines.extend(self.smi.stdout), daemon=True)
            self.thread.start()
        except Exception:
            self.smi = None

    def stop(self) -> dict:
        """{"sm_mhz": median, "sm_max_mhz", "reasons": [...], "samples", "source"} for this rank's GPU."""
        self.stop_flag = True
        if self.smi is not None:
            self.smi.terminate()
            self.thread.join(timeout=2)
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            reasons = set()
            for ln in self.lines:
                f = [x.strip() for x in ln.split(",")]
                try:
                    self.mhz.append(float(f[0])); self.max_mhz = float(f[1])
                except (ValueError, IndexError):
                    continue
                reasons |= {n for n, v in zip(names, f[2:6]) if v.lower().startswith("active")}
            src = "nvidia-smi"
        elif self.thread is not None:
            self.thread.join(timeout=2)
            reasons = {n for n, bit in self.REASONS.items() if self.mask & bit}
            src = "nvml"
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock query unavailable"], "samples": 0, "source": None}
        return {"sm_mhz": statistics.median(self.mhz) if self.mhz else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(reasons), "samples": len(self.mhz), "source": src}


def merge_clocks(per_rank: list) -> dict:
    """One "clocks" object for the JSON line: the slowest GPU's median sets the pace of a sharded step."""
    ok = [c for c in per_rank if c and c.get("sm_mhz") is not None]
    if not ok:
        return per_rank[0] if per_rank and per_rank[0] else {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock query unavailable"]}
    out = {"sm_mhz": min(c["sm_mhz"] for c in ok), "sm_max_mhz": max(c["sm_max_mhz"] or 0 for c in ok) or None,
           "reasons": sorted(set().union(*[set(c["reasons"]) for c in ok])), "samples": sum(c["samples"] for c in ok),
           "source": ok[0]["source"]}
    if len(per_rank) > 1:
        out["per_gpu_sm_mhz"] = [c["sm_mhz"] if c else None for c in per_rank]
    return out


def host_threads() -> int:
    """Threads for the CPU legs: the cores this process may actually use (affinity and cgroup quota), then a
    short calibration over power-of-two counts -- oversubscribing a quota-limited container is slower."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    cands = sorted({c for c in (n, 64, 32, 16, 8) if 1 <= c <= n})
    if len(cands) == 1:
        return cands[0]
    a = torch.randn(8, 64, 96, 128)
    w = torch.randn(64, 64, 3, 3)
    m = torch.randn(2048, 512)
    best, best_t = cands[-1], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        torch.nn.functional.conv2d(a, w, padding=1); m @ m.t()
        t0 = time.perf_counter()
        for _ in range(3):
            torch.nn.functional.conv2d(a, w, padding=1); m @ m.t()
        dt = time.perf_counter() - t0
        if dt < best_t * 0.95:
            best, best_t = c, dt
    return best


def make_inputs(n_global: int):
    """Synthetic clip + queries for the CUDA arm (product-side generators; the oracle is not involved)."""
    from pips_b200 import synthetic
    rgbs = synthetic.smooth_video(B, S, H, W, seed=1234).to(torch.bfloat16)       # integers 0..255: exact in bf16
    xys = synthetic.random_queries(B, n_global, H, W, seed=4321)
    return rgbs, xys


def make_oracle_inputs():
    """Same-shaped workload for the CPU legs, from the oracle's own generators and seeded weights."""
    from oracle import pips_oracle as po
    return (po.init_state_dict(seed=0, head_scale=0.05), po.smooth_video(B, S, H, W, seed=1234),
            po.random_queries(B, N_PER_GPU, H, W, seed=4321))


# ------------------------------------------------------------------------------------------ reference arm
def workload_name(world: int) -> str:
    """config.workload of BOTH arms: the BASELINE configuration the metric is quoted on."""
    return (f"BASELINE cfg2 per GPU: B={B}, S={S}, {H}x{W} bf16 video, N={N_PER_GPU}/GPU (global N={N_PER_GPU * world}), "
            f"iters={ITERS}, stride={STRIDE}")


def run_reference(args, rank, world):
    """The reference's algorithm (all-pairs volume, dense heat-map, fp32 torch ops -- nets/pips.py:428-611
    restated in oracle/pips_oracle.py; the reference itself is Python and cannot travel to the GPU box) on
    the host CPU cores, on a bounded sample of the same workload."""
    if rank != 0:
        return
    from oracle import pips_oracle as po
    cores = host_threads()
    torch.set_num_threads(cores)
    sd, rgbs, xys = make_oracle_inputs()
    bs, ns = 1, 256                                # reference-style chunk (test_on_davis.py:111-125 chunks N by 256)
    rg, xy = rgbs[:bs].float(), xys[:bs, :ns]

    def step():
        with torch.no_grad():
            return po.forward(sd, xy, rg, iters=ITERS, stride=STRIDE, allpairs=True, faithful_dead_work=True)

    steps, warm = args.steps, args.warmup
    for _ in range(warm):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = step()
    dt = (time.perf_counter() - t0) / steps
    if args.dump_outputs:
        dump_outputs(out, args.dump_outputs)
    val = bs * S * ns * ITERS / dt
    sample = f"B={bs} of {B}, N={ns} of {N_PER_GPU}, iters={ITERS}, incl. fnet, all-pairs volume + dense heat-map as the reference computes them"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(world), "sample_per_step": sample, "stride": STRIDE},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------ our arm
def cpu_baseline_leg():
    from oracle import pips_oracle as po
    cores = host_threads()
    torch.set_num_threads(cores)
    sd, rgbs, xys = make_oracle_inputs()
    bs, ns = 1, 256
    rg, xy = rgbs[:bs].float(), xys[:bs, :ns]
    with torch.no_grad():
        po.forward(sd, xy, rg, iters=1, stride=STRIDE, allpairs=True)          # warm caches / threads
        t0 = time.perf_counter()
        reps = 0
        while reps < 2 or (time.perf_counter() - t0 < 10.0 and reps < 8):
            po.forward(sd, xy, rg, iters=ITERS, stride=STRIDE, allpairs=True, faithful_dead_work=True)
            reps += 1
        dt = (time.perf_counter() - t0) / reps
    return {"value": bs * S * ns * ITERS / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"B={bs} of {B}, N={ns} of {N_PER_GPU}, iters={ITERS}, {reps} forwards incl. fnet, reference algorithm (all-pairs volume + dense heat-map)"}


DUMP_BYTES = 63 * 10**6                   # array data; with the .npy headers the files stay under 64 MB


def dump_outputs(out, directory: str) -> None:
    """What ``Pips.forward`` handed its caller, as float32 ``<name>.npy`` in ``directory``: coord_predictions
    (iters,B,S,N,2), coord_predictions2 (iters+4,B,S,N,2) and vis_e (B,S,N).  When they hold more than DUMP_BYTES,
    every k-th particle is written (the smallest k that fits), the same particles in every array."""
    import numpy as np
    preds, preds2, vis_e, _ = out
    arrays = {"coord_predictions": (torch.stack(preds), 3), "coord_predictions2": (torch.stack(preds2), 3), "vis_e": (vis_e, 2)}
    n = vis_e.shape[2]
    per_particle = sum(a.numel() // n * 4 for a, _ in arrays.values())
    every = -(-n // max(1, DUMP_BYTES // per_particle))
    os.makedirs(directory, exist_ok=True)
    for name, (a, dim) in arrays.items():
        keep = torch.arange(0, n, every, device=a.device)
        np.save(os.path.join(directory, name + ".npy"), a.index_select(dim, keep).float().cpu().numpy())


def _stats(per_ms: list) -> dict:
    return {"min": round(min(per_ms), 3), "median": round(statistics.median(per_ms), 3), "max": round(max(per_ms), 3),
            "stdev": round(statistics.pstdev(per_ms), 3), "n": len(per_ms)}


def time_config(model, dev, world, *, Bc, Hc, Wc, n_global, stride, steps=5, warm=3, seed=3):
    """One more BASELINE configuration through the same public call: device-resident loop and pinned-host loop,
    CUDA events per step, L2 flushed before each step, max over ranks.  ``model`` carries the stride / sharding."""
    import torch.distributed as dist
    from pips_b200 import synthetic
    rgbs_h = synthetic.smooth_video(Bc, S, Hc, Wc, seed=seed).to(torch.bfloat16).pin_memory()
    xys_h = synthetic.random_queries(Bc, n_global, Hc, Wc, seed=seed + 1).pin_memory()
    rgbs, xys = rgbs_h.to(dev), xys_h.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run(step):
        per = []
        evs = []
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); step(); e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        per = [a.elapsed_time(b) for a, b in evs]
        t = torch.tensor([sum(per) / steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), per

    def step_device():
        with torch.no_grad():
            return model(xys, rgbs, iters=ITERS)

    def step_host():
        with torch.no_grad():
            out = model(xys_h.to(dev, non_blocking=True), rgbs_h.to(dev, non_blocking=True), iters=ITERS)
            return out[0][-1].cpu(), out[2].cpu()

    for _ in range(warm):
        out = step_device()
    finite = bool(torch.isfinite(out[0][-1]).all())
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms_dev, per_dev = run(step_device)
    step_host()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms_e2e, per_e2e = run(step_host)
    upd = Bc * S * n_global * ITERS
    return {"workload": f"B={Bc}, S={S}, {Hc}x{Wc} bf16 video, global N={n_global}, iters={ITERS}, stride={stride}, {world} GPU(s)",
            "value": upd / (ms_dev * 1e-3), "unit": UNIT, "ms_per_step": ms_dev, "steps": steps, "finite": finite,
            "e2e": {"value": upd / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": rgbs_h.numel() * rgbs_h.element_size() + xys_h.numel() * 4,
                    "d2h_bytes_per_step": (Bc * S * n_global * 3) * 4},
            "ms_per_step_stats_rank0": _stats(per_dev)}


def corr_nonresident_block(dev, feat, pk):
    """corr_gather where the HBM roofline means something: a pyramid that does NOT fit the 126 MB L2 (BASELINE cfg 5's
    clip: 100 frames of 90x160 maps at stride 4, 0.98 GB in fp32), 4096 tracks reading their own 8-frame windows
    (chained-tracking addressing), L2 flushed before every launch.  Both byte counts are given: SURVEY 8d's 66 440 B per
    unit (bf16 pyramid + bf16 row) and what this configuration actually moves (fp32 pyramid, (hi, lo) row)."""
    from pips_b200 import _lib as L
    from pips_b200.engine import Pyramid
    lib = L.load()
    fdt = L.FEAT_DTYPES[feat]
    Bc, T, Nc, H8, W8 = 1, 100, 4096, 90, 160
    g = torch.Generator(device=dev).manual_seed(7)
    fm = torch.randn(Bc * T, 128, H8, W8, device=dev, generator=g)
    pyr = Pyramid(Bc * T, H8, W8, fdt, dev)
    st = torch.cuda.current_stream().cuda_stream
    pyr.build(fm, st)
    del fm
    coords = torch.rand(Bc, S, Nc, 2, device=dev, generator=g) * torch.tensor([W8 - 1.0, H8 - 1.0], device=dev)
    ffeats = torch.randn(Bc * Nc, S, 128, device=dev, generator=g)
    times = torch.linspace(0, S, S, device=dev)
    fb = torch.randint(0, T - 8, (Bc, Nc), device=dev, dtype=torch.int32, generator=g)
    M = Bc * Nc * S
    x_hi = torch.empty(M, 576, dtype=torch.bfloat16, device=dev)
    x_lo = torch.empty_like(x_hi)
    lvl = L.ptr_array(pyr.levels())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run():
        L.check(lib.pips_corr_gather(lvl, fdt, Bc, S, Nc, H8, W8, L.ptr(coords), L.ptr(ffeats), L.ptr(times), L.ptr(fb), T,
                                     L.ptr(x_hi), L.ptr(x_lo), None, 576, st))
    for _ in range(3):
        run()
    ts = []
    for _ in range(10):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); run(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ms = statistics.median(ts)
    e_f = 4 if feat == "fp32" else 2
    b_actual, b_survey = 4 * 64 * 128 * e_f + 128 * 4 + 576 * 4, 66440
    pyr_mb = sum(t.numel() * t.element_size() for t in pyr.levels()) / 1e6
    return {"kernel": "corr_gather_kernel", "bound": "hbm", "workload": f"{T} frames of {H8}x{W8} maps ({pyr_mb:.0f} MB pyramid, > L2), {Nc} tracks x 8 frames",
            "ms_per_launch": ms, "units": M, "unit": "GB/s", "peak": pk["hbm_gbs"], "peak_source": pk["source"] + " (copy bandwidth)",
            "achieved": b_survey * M / (ms * 1e-3) / 1e9, "bytes_per_unit": b_survey, "frac": b_survey * M / (ms * 1e-3) / 1e9 / pk["hbm_gbs"],
            "achieved_actual_bytes": b_actual * M / (ms * 1e-3) / 1e9, "bytes_per_unit_actual": b_actual,
            "note": "algorithmic gather bytes; patches of neighbouring tracks overlap, so part of them is served by L2 even here"}


def chain_block(dev, precision, feat):
    """BASELINE cfg 5: chained tracking over a 100-frame 360x640 clip, N=512, 8-frame windows, stride 4, one GPU
    (chain_demo.py:40-83 semantics; all particles advance together, pips_b200/chain.py)."""
    from pips_b200 import synthetic
    from pips_b200.chain import track_chain
    T, Hc, Wc, Nc = 100, 360, 640, 512
    rgbs = synthetic.smooth_video(1, T, Hc, Wc, seed=99).to(dev)
    xy0 = synthetic.random_queries(1, Nc, Hc, Wc, seed=98).to(dev)
    model = synthetic.seeded_model(stride=4, precision=precision, feat_dtype=feat).to(dev).eval()
    out = {"workload": f"{T}x{Hc}x{Wc} clip, N={Nc}, 8-frame windows, iters={ITERS}, stride 4, 1 GPU", "unit": "tracked particle-frames/s"}
    for key, adv in (("visibility_driven", None), ("fixed_advance_7", 7)):
        for _ in range(2):
            track_chain(model, rgbs, xy0, iters=ITERS, advance=adv)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        trajs, rounds = track_chain(model, rgbs, xy0, iters=ITERS, return_rounds=True, advance=adv)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        # every round refines 8 frames of each still-active track; the fixed schedule makes that count data-independent
        out[key] = {"rounds": rounds, "ms": ms, "value": T * Nc / (ms * 1e-3), "finite": bool(torch.isfinite(trajs).all()),
                    "includes": "fnet of all 100 frames once + pyramid + every round's 6 iterations"}
    return out


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from pips_b200 import synthetic

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    n_global = N_PER_GPU * world
    rgbs_h, xys_h = make_inputs(n_global)
    model = synthetic.seeded_model(stride=STRIDE, seed=0, head_scale=0.05, precision=args.precision, feat_dtype=args.feat).to(dev).eval()
    if world > 1:
        model.shard_particles()
    rgbs_h, xys_h = rgbs_h.pin_memory(), xys_h.pin_memory()
    rgbs, xys = rgbs_h.to(dev), xys_h.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)             # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        with torch.no_grad():
            return model(xys, rgbs, iters=ITERS)

    def step_host():
        with torch.no_grad():
            out = model(xys_h.to(dev, non_blocking=True), rgbs_h.to(dev, non_blocking=True), iters=ITERS)
            return out[0][-1].cpu(), out[2].cpu()

    def timed(step, k):
        """k steps, L2 flushed before each; returns (total seconds, [ms per step], output of the last step) from CUDA
        events on this stream."""
        evs, out = [], None
        for _ in range(k):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); out = step(); e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        per = [a.elapsed_time(b) for a, b in evs]
        return sum(per) / 1e3, per, out

    # sharded runs: the particle shares become speed-weighted after the 5th forward (pips_b200/sharding.py::_Balance) and the
    # next forward re-captures its CUDA graph at the new share -- all of that belongs to the warm-up
    n_warm = max(3, args.warmup) if world == 1 else max(8, args.warmup)
    # The clock sampler is started BEFORE the warm-up: NVML initialisation in 8 processes at once stalls the driver for
    # ~0.1 s, and when that fell into the first timed step (round 1 / r02i: one 120 ms step among twenty 38 ms ones) the
    # device-timed mean came out above the e2e mean.  Samples taken during the warm-up are dropped by mark().
    sampler = ClockSampler(dev)                      # every rank watches its own GPU
    sampler.start()
    for _ in range(n_warm):
        step_device()
    barrier()
    sampler.mark()
    t_dev, per_dev, last = timed(step_device, args.steps)
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(last, args.dump_outputs)
    if world > 1:
        all_clocks = [None] * world
        dist.all_gather_object(all_clocks, clocks)
    else:
        all_clocks = [clocks]
    clocks = merge_clocks(all_clocks)
    from pips_b200 import encoder_fast
    launches = (model.engine.launches + (encoder_fast.LAUNCHES[0] if model.fnet_mode == 'tc' else 0)) * args.steps
    step_host()
    barrier()
    t_e2e, per_e2e, _ = timed(step_host, args.steps)
    barrier()
    if world > 1:
        t = torch.tensor([t_dev, t_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_dev, t_e2e = t.tolist()

    # ---- the other BASELINE configurations, through the same call (every rank takes part in the sharded ones)
    extra = {}
    if not args.no_extra:
        def guarded(name, fn):
            try:
                extra[name] = fn()
            except Exception as e:                      # noqa: BLE001 -- a failed extra block must not lose the main line
                extra[name] = {"error": f"{type(e).__name__}: {e}"[:300]}

        def fresh(stride):
            m = synthetic.seeded_model(stride=stride, seed=0, head_scale=0.05, precision=args.precision, feat_dtype=args.feat).to(dev).eval()
            if world > 1:
                m.shard_particles()
                m._balance = model._balance             # the GPUs' measured rates carry over: no second calibration
            return m

        if world == 1:
            if N_PER_GPU != 4096:
                # the north-star target configuration: S=8, 384x512, N=4096, iters=6 on ONE B200 (>= 1 M updates/s asked)
                guarded("n4096_1gpu", lambda: time_config(model, dev, 1, Bc=B, Hc=H, Wc=W, n_global=4096, stride=STRIDE, seed=1234))
            guarded("cfg1_demo_shape_1gpu", lambda: time_config(fresh(4), dev, 1, Bc=1, Hc=360, Wc=640, n_global=256, stride=4, steps=10))
            guarded("cfg4_1gpu", lambda: time_config(fresh(8), dev, 1, Bc=1, Hc=720, Wc=1280, n_global=16384, stride=8))
            guarded("cfg5_chain_1gpu", lambda: chain_block(dev, args.precision, args.feat))
        else:
            # BASELINE cfg 3 as stated: FIXED N=4096 sharded over the ranks (strong scaling; the main line is weak scaling)
            guarded("strong_cfg3", lambda: time_config(model, dev, world, Bc=B, Hc=H, Wc=W, n_global=4096, stride=STRIDE, seed=1234))
            # BASELINE cfg 4: 8 x 720 x 1280, N=16384, B=1, particle-sharded (frames of the encoder sharded as well)
            guarded("cfg4_sharded", lambda: time_config(fresh(8), dev, world, Bc=1, Hc=720, Wc=1280, n_global=16384, stride=8))
    if rank != 0:
        return

    updates = B * S * n_global * ITERS
    pk = peaks()
    shard_sizes_now = None
    if world > 1 and getattr(model, "_balance", None) is not None and model._balance.weights:
        from pips_b200.sharding import shard_sizes
        shard_sizes_now = shard_sizes(n_global, model._balance.weights)
    # per-kernel timing of one iteration, live, same buffers (CUDA events around every launch)
    REPS = 6
    with torch.no_grad():
        for _ in range(12):                       # ~0.5 s of back-to-back forwards: the per-kernel timings below are taken in the
            model(xys, rgbs, iters=ITERS)         # power-capped steady state of a long step, not at the boost clock of a cold burst
        fmaps = model.encode(rgbs)
        coords = (xys[:, :N_PER_GPU] / STRIDE).reshape(B, 1, N_PER_GPU, 2).repeat(1, S, 1, 1)
        prof, dims = model.engine.profile_iteration(model, fmaps.float(), coords, STRIDE, reps=REPS)
    # the encoder alone (its CUDA graph), same inputs, L2 flushed before each replay
    fnet_ms = []
    with torch.no_grad():
        for _ in range(2):
            model.encode(rgbs)
        for _ in range(8):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); model.encode(rgbs); e1.record(); torch.cuda.synchronize()
            fnet_ms.append(e0.elapsed_time(e1))
    mean = {k: statistics.mean(v) for k, v in prof.items()}
    per_iter = {k: sum(v) / REPS for k, v in prof.items()}
    M = dims["M"]
    gemm_ms = per_iter["gemm_fc1"] + per_iter["gemm_fc2"]
    gemm_flop = 2.0 * M * 2048 * 512 * 2 * 12
    achieved_tf = gemm_flop / (gemm_ms * 1e-3) / 1e12
    tc = args.precision != "fp32"
    mma_per_product = 3 if args.precision == "bf16x3" else 1
    roofline = {"kernel": "gemm_tc2_kernel (tcgen05 cta_group::2; FC1+FC2 of the 12 channel-mixing blocks)" if tc else "gemm_f32_kernel",
                "bound": "tensor", "achieved": achieved_tf, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": achieved_tf / pk["bf16_tflops_sustained"], "traffic": None,
                "peak_source": pk["source"] + " (sustained bf16 cuBLAS)", "share_of_iteration": gemm_ms / sum(per_iter.values()),
                "mma_issued_frac": achieved_tf * mma_per_product / pk["bf16_tflops_sustained"] if tc else None}
    e_f = 4 if args.feat == "fp32" else 2
    e_o = {"fp32": 4, "bf16x3": 4, "bf16": 2}[args.precision]
    unit_bytes = 4 * 64 * 128 * e_f + 128 * 4 + 576 * e_o
    corr_gbs = unit_bytes * (M) / (mean["corr_gather"] * 1e-3) / 1e9
    roofline_corr = {"kernel": "corr_gather_kernel", "bound": "hbm", "achieved": corr_gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                     "frac": corr_gbs / pk["hbm_gbs"], "traffic": None, "bytes_per_unit": unit_bytes,
                     "frac_survey_bytes": 66440 * M / (mean["corr_gather"] * 1e-3) / 1e9 / pk["hbm_gbs"],
                     "peak_source": pk["source"] + " (copy bandwidth)",
                     "note": "the 67 MB pyramid is L2-resident at this configuration: algorithmic gather bytes over the kernel time exceed the "
                             "HBM copy peak and are NOT an HBM fraction -- roofline_corr_hbm measures the kernel on a pyramid larger than L2"}
    # DRAM bytes per launch come from an `ncu --set full` capture (tools/ncu_traffic.py writes the file together with the
    # digest of the kernel sources it profiled); they are reported only when that digest is the library's that runs now.
    try:
        from pips_b200 import _build
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            tr = json.load(f)
        if tr.get("source_digest") == _build.source_digest():
            roofline["traffic"] = tr.get("gemm_fc_bytes_per_launch")
            roofline_corr["traffic"] = tr.get("corr_gather_bytes_per_launch")
            roofline["traffic_source"] = roofline_corr["traffic_source"] = tr.get("source")
        else:
            roofline["traffic_source"] = roofline_corr["traffic_source"] = "profiles/ncu_traffic.json is from other kernel sources: not reported"
    except Exception:
        pass
    corr_hbm = None
    if world == 1 and not args.no_extra:
        try:
            corr_hbm = corr_nonresident_block(dev, args.feat, pk)
        except Exception as e:                          # noqa: BLE001
            corr_hbm = {"error": f"{type(e).__name__}: {e}"[:300]}
    eager = None
    if world == 1 and not args.no_eager:
        # the reference's algorithm as eager torch ops on THIS GPU (all-pairs volume, dense heat-map, strict-fp32
        # cuDNN/cuBLAS) -- pips_b200/torch_path.py, which is pinned to the reference's outputs on CPU.  Context only.
        from pips_b200.torch_path import forward_torch
        mode = model.fnet_mode
        model.fnet_mode = "plain"
        with torch.no_grad():
            for _ in range(2):
                forward_torch(model, xys, rgbs.float(), iters=ITERS)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                forward_torch(model, xys, rgbs.float(), iters=ITERS)
            e1.record(); torch.cuda.synchronize()
        model.fnet_mode = mode
        eager = {"value": updates / (e0.elapsed_time(e1) / 3e3), "unit": UNIT, "ms_per_step": e0.elapsed_time(e1) / 3,
                 "what": "reference algorithm as eager torch ops on the same B200 (fp32, TF32 off)"}
    cpu = cpu_baseline_leg() if world == 1 and not args.no_cpu_baseline else None
    h2d = rgbs_h.numel() * rgbs_h.element_size() + xys_h.numel() * 4
    d2h = (B * S * n_global * 2 + B * S * n_global) * 4
    line = {"metric": METRIC, "value": updates / (t_dev / args.steps), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {"fp32": "f32", "bf16x3": "bf16x3 (hi/lo split, fp32 accumulate) + f32", "bf16": "bf16"}[args.precision],
            "data": "synthetic",
            "config": {"workload": workload_name(world),
                       "precision": args.precision, "feat_dtype": args.feat, "parallelism": (f"particle-sharded dp{world}, shares " + ("speed-weighted " + str(shard_sizes_now) if shard_sizes_now else "equal")) if world > 1 else "single GPU",
                       "includes": "fnet (tcgen05 convs) + pyramid + 6 refinement iterations + vis head", "fnet_mode": model.fnet_mode, "l2": "256 MB write between steps (L2 flushed); working set > L2"},
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": updates / (t_e2e / args.steps), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": t_e2e / args.steps * 1e3},
            "roofline": roofline, "roofline_corr": roofline_corr,
            "kernel_ms_per_iteration": {k: round(v, 4) for k, v in per_iter.items()},
            "fnet_ms": {"median": round(statistics.median(fnet_ms), 3), "min": round(min(fnet_ms), 3), "frames": B * S,
                        "what": "BasicEncoder on all B*S frames of this rank's batch (unsharded), one CUDA-graph replay"},
            "loop_only": {"ms_per_iteration": sum(per_iter.values()), "updates_per_s": B * S * N_PER_GPU / (sum(per_iter.values()) * 1e-3)},
            "whole_path_tensor_frac": (updates * UNIT_FLOP / (t_dev / args.steps)) / 1e12 / pk["bf16_tflops_sustained"] / world}
    line["ms_per_step_stats_rank0"] = {"device_loop": _stats(per_dev), "e2e_loop": _stats(per_e2e)}
    line.update(extra)
    if corr_hbm is not None:
        line["roofline_corr_hbm"] = corr_hbm
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if eager is not None:
        line["torch_eager_same_gpu"] = eager
    emit(line)


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The one JSON line goes to the real stdout; everything else (NCCL banners, warnings) was rerouted."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                                  # libraries that print to fd 1 (NCCL version banner) -> stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("PIPS_B200_PRECISION", "bf16x3"), choices=["fp32", "bf16x3", "bf16"])
    ap.add_argument("--feat", default=os.environ.get("PIPS_B200_FEAT", "fp32"), choices=["fp32", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager", action="store_true", help="skip the eager-torch restatement of the reference on this GPU")
    ap.add_argument("--no-extra", action="store_true", help="skip the other BASELINE configurations (n4096_1gpu, cfg1/4/5, strong_cfg3, cfg4_sharded)")
    ap.add_argument("--particles", type=int, default=0, help="particles per GPU (default 1024 = BASELINE cfg2; 4096 = cfg3 on one GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as float32 DIR/<name>.npy "
                                                            "(inputs are seeded: runs with the same arguments are comparable)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.particles > 0:
        global N_PER_GPU
        N_PER_GPU = args.particles
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
