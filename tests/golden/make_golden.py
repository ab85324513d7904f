"""Generate golden vectors from the UNMODIFIED reference (a checkout of aharley/pips).

    python tests/golden/make_golden.py --reference DIR [--cfg2 | --cfg4 | --demo | --nets-layout]

The tests import only the case definitions and input generators below; they never need the reference.

The reference (aharley/pips, nets/pips.py) is imported as-is; the only shim is
``torch.Tensor.cuda = identity`` because nets/pips.py:429 calls ``.cuda()`` on a
scalar that is never used (SURVEY.md section 0-4).  Weights come from
``oracle.pips_oracle.init_state_dict`` and are loaded with ``strict=True``, which
also pins the state_dict key/shape contract of SURVEY.md section 8b.  Inputs are
regenerated from seeds by the tests, so only outputs are stored.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import pips_oracle as po  # noqa: E402

CASES = {
    # name: dict(B, H, W, N, stride, iters, head_scale, seed, oob, warm)
    "tiny_s8": dict(B=1, H=128, W=128, N=12, stride=8, iters=3, head_scale=0.05, seed=1, oob=False, warm=False),
    "rect_s4_oob": dict(B=2, H=128, W=192, N=20, stride=4, iters=6, head_scale=0.05, seed=2, oob=True, warm=False),
    "odd_s8": dict(B=1, H=184, W=360, N=16, stride=8, iters=4, head_scale=0.02, seed=3, oob=True, warm=False),
    "warm_s8": dict(B=1, H=128, W=160, N=10, stride=8, iters=2, head_scale=0.05, seed=4, oob=False, warm=True),
    "undamped_1it": dict(B=1, H=128, W=128, N=8, stride=8, iters=1, head_scale=1.0, seed=5, oob=False, warm=False),
}


# Oracle-only pins (CPU tests): the demo configuration's sizes (BASELINE cfg 1: 8 x 360 x 640, stride 4, 6 iterations;
# 90 x 160 feature maps, odd pyramid sizes 45 -> 22 -> 11) -- the -m gpu suite checks the CUDA path against the live
# oracle at exactly this shape, this pins the oracle at this shape to the reference.
CPU_CASES = {
    "demo_s4": dict(B=1, H=360, W=640, N=24, stride=4, iters=6, head_scale=0.05, seed=8, oob=True, warm=False),
}


LOSS_CASE = dict(B=2, H=128, W=128, N=9, stride=8, iters=3, head_scale=0.05, seed=6, oob=False, warm=False)


FCP_SEL = [0, 4, 7]          # particles whose dense score maps (nets/pips.py:504-511) are recorded for LOSS_CASE


def loss_targets(c, xys):
    g = torch.Generator().manual_seed(400 + c["seed"])
    trajs_g = xys[:, None] + torch.cumsum(torch.randn(c["B"], 8, c["N"], 2, generator=g), 1)
    vis_g = (torch.rand(c["B"], 8, c["N"], generator=g) > 0.3).float()
    valids = (torch.rand(c["B"], 8, c["N"], generator=g) > 0.1).float()
    return trajs_g, vis_g, valids


CHAIN_CASE = dict(T=19, H=96, W=128, N=5, stride=4, iters=6, head_scale=0.05, seed=7)


def chain_inputs(c):
    rgbs = po.smooth_video(1, c["T"], c["H"], c["W"], seed=500 + c["seed"])
    xy0 = po.random_queries(1, c["N"], c["H"], c["W"], seed=600 + c["seed"])
    return rgbs, xy0


def case_inputs(c):
    """Shared with tests/: deterministic inputs for a golden case."""
    rgbs = po.smooth_video(c["B"], 8, c["H"], c["W"], seed=100 + c["seed"])
    xys = po.random_queries(c["B"], c["N"], c["H"], c["W"], seed=200 + c["seed"])
    if c["oob"]:
        # push a few queries onto / across the border: exercises zero padding in the
        # correlation sampler and index clamping in the initial feature gather
        xys[:, 0] = torch.tensor([0.0, 0.0])
        xys[:, 1] = torch.tensor([c["W"] - 1.0, c["H"] - 1.0])
        xys[:, 2] = torch.tensor([-5.5, 17.25])
        xys[:, 3] = torch.tensor([c["W"] + 3.0, c["H"] + 6.5])
        xys[:, 4] = torch.tensor([float(c["stride"] * 5), float(c["stride"] * 7)])   # exact integer grid coords
    extra = {}
    if c["warm"]:
        g = torch.Generator().manual_seed(300 + c["seed"])
        drift = torch.cumsum(torch.randn(c["B"], 8, c["N"], 2, generator=g) * 1.5, 1)
        extra["coords_init"] = xys[:, None] + drift - drift[:, :1]
        extra["feat_init"] = torch.randn(c["B"], c["N"], 128, generator=g) * 0.5
    return rgbs, xys, extra


def main():
    torch.Tensor.cuda = lambda self, *a, **k: self
    from nets.pips import Pips  # the reference, unmodified

    torch.set_num_threads(8)
    out = {}
    for name, c in list(CASES.items()) + list(CPU_CASES.items()):
        sd = po.init_state_dict(seed=c["seed"], head_scale=c["head_scale"])
        model = Pips(S=8, stride=c["stride"]).eval()
        model.load_state_dict(sd, strict=True)
        rgbs, xys, extra = case_inputs(c)
        with torch.no_grad():
            preds, preds2, vis_e, ffeat, losses = model(xys, rgbs, iters=c["iters"], return_feat=True, **extra)
        assert losses is None and len(preds2) == c["iters"] + 4
        out[name + "/preds"] = torch.stack(preds).numpy()
        out[name + "/vis_e"] = vis_e.numpy()
        out[name + "/ffeat"] = ffeat.numpy()
        print(name, "trajs_e range", float(preds[-1].min()), float(preds[-1].max()),
              "mean |d| from init", float((preds[-1] - xys[:, None]).abs().mean()))
    # supervised call (nets/pips.py:600-606): losses + is_train semantics, consumed by the torch path tests
    for name, is_train in (("loss_s8", False), ("train_s8", True)):
        c = LOSS_CASE
        sd = po.init_state_dict(seed=c["seed"], head_scale=c["head_scale"])
        model = Pips(S=8, stride=c["stride"]).eval()
        model.load_state_dict(sd, strict=True)
        rgbs, xys, extra = case_inputs(c)
        trajs_g, vis_g, valids = loss_targets(c, xys)
        import nets.pips as ref_mod
        seen, real_loss = {}, ref_mod.score_map_loss

        def spy(fcps, *a, **k):                      # fcps is only visible as this loss's argument (nets/pips.py:603)
            seen["fcps"] = fcps.detach().clone()
            return real_loss(fcps, *a, **k)

        ref_mod.score_map_loss = spy
        try:
            with torch.no_grad():
                preds, _, vis_e, losses = model(xys, rgbs, iters=c["iters"], trajs_g=trajs_g, vis_g=vis_g, valids=valids, is_train=is_train)
        finally:
            ref_mod.score_map_loss = real_loss
        if not is_train:
            out[name + "/fcps_sel"] = seen["fcps"][:, :, :, FCP_SEL].numpy()      # (B,S,I,3,H8,W8)
        out[name + "/preds"] = torch.stack(preds).numpy()
        out[name + "/vis_e"] = vis_e.numpy()
        out[name + "/losses"] = np.array([float(l) for l in losses], dtype=np.float64)
        print(name, "losses", out[name + "/losses"])
    # edge case: no particles.  The reference does not return empty results, it fails -- record how.
    model = Pips(S=8, stride=8).eval()
    try:
        with torch.no_grad():
            model(torch.zeros(2, 0, 2), torch.zeros(2, 8, 3, 64, 64), iters=2)
        out["edge/n0_error"] = np.array("none")
    except Exception as e:                                             # noqa: BLE001
        out["edge/n0_error"] = np.array(type(e).__name__)
    print("N = 0 ->", out["edge/n0_error"])
    # chained long-video tracking (chain_demo.py:40-83) with the reference model as the 8-frame tracker
    c = CHAIN_CASE
    sd = po.init_state_dict(seed=c["seed"], head_scale=c["head_scale"])
    model = Pips(S=8, stride=c["stride"]).eval()
    model.load_state_dict(sd, strict=True)
    rgbs, xy0 = chain_inputs(c)

    def ref_window(xys, seq, feat_init):
        with torch.no_grad():
            o = model(xys, seq, iters=c["iters"], feat_init=feat_init, return_feat=True)
        return o[0], o[2], o[3]

    trajs, skips = po.chain_track(ref_window, rgbs, xy0, iters=c["iters"])
    out["chain/trajs"] = trajs.numpy()
    out["chain/skips"] = np.array([len(h) for h in skips] + [s for h in skips for s in h], dtype=np.int64)
    print("chain skips", skips)
    np.savez_compressed(os.path.join(HERE, "reference_outputs.npz"), **out)
    print("wrote", os.path.join(HERE, "reference_outputs.npz"))


# BASELINE cfg 2 at full size (the bench workload): B=4, 8 x 384 x 512, N=1024, stride 8, 6 iterations.  Recorded once
# (minutes of CPU time, ~10 GB of score maps inside the reference) into its own file; stored subsampled to stay small:
# every iteration's prediction for every 4th particle, the final prediction and the visibility logits for all.
CFG2_CASE = dict(B=4, H=384, W=512, N=1024, stride=8, iters=6, head_scale=0.05, seed=9, oob=False, warm=False)
CFG2_EVERY = 4


def main_cfg2():
    torch.Tensor.cuda = lambda self, *a, **k: self
    from nets.pips import Pips  # the reference, unmodified

    torch.set_num_threads(min(16, os.cpu_count() or 1))
    c = CFG2_CASE
    sd = po.init_state_dict(seed=c["seed"], head_scale=c["head_scale"])
    model = Pips(S=8, stride=c["stride"]).eval()
    model.load_state_dict(sd, strict=True)
    rgbs, xys, _ = case_inputs(c)
    with torch.no_grad():
        preds, _, vis_e, ffeat, _ = model(xys, rgbs, iters=c["iters"], return_feat=True)
    p = torch.stack(preds)                                             # (6, B, S, N, 2)
    out = {"preds_sub": p[:, :, :, ::CFG2_EVERY].numpy(), "preds_final": p[-1].numpy(), "vis_e": vis_e.numpy(),
           "ffeat_sub": ffeat[:, ::16].numpy()}
    np.savez_compressed(os.path.join(HERE, "reference_cfg2.npz"), **out)
    print("cfg2: mean |d| from init", float((p[-1] - xys[:, None]).abs().mean()), "max", float((p[-1] - xys[:, None]).abs().max()))
    print("wrote", os.path.join(HERE, "reference_cfg2.npz"), os.path.getsize(os.path.join(HERE, "reference_cfg2.npz")), "bytes")


# BASELINE cfg 4 shape: B=1, 8 x 720 x 1280, stride 8 (90 x 160 maps -> 45x80 -> 22x40 -> 11x20), N=16384 queries, 6 iterations.
# The reference cannot hold the all-pairs volume for 16384 particles (10 GB per iteration); its own recipe for many
# particles is to run them in chunks of 256 (test_on_davis.py:111-125).  Particles are independent (nets/pips.py:517-524),
# so ONE such chunk -- every 64th query of the 16384 -- pins the CUDA path at this shape: the GPU test tracks all 16384
# and compares those 256.
CFG4_CASE = dict(B=1, H=720, W=1280, N=16384, stride=8, iters=6, head_scale=0.05, seed=10, oob=False, warm=False)
CFG4_EVERY = 64


def main_cfg4():
    torch.Tensor.cuda = lambda self, *a, **k: self
    from nets.pips import Pips  # the reference, unmodified

    torch.set_num_threads(min(16, os.cpu_count() or 1))
    c = CFG4_CASE
    sd = po.init_state_dict(seed=c["seed"], head_scale=c["head_scale"])
    model = Pips(S=8, stride=c["stride"]).eval()
    model.load_state_dict(sd, strict=True)
    rgbs, xys, _ = case_inputs(c)
    chunk = xys[:, ::CFG4_EVERY].contiguous()                          # (1, 256, 2)
    assert chunk.shape[1] == 256
    with torch.no_grad():
        preds, _, vis_e, ffeat, _ = model(chunk, rgbs, iters=c["iters"], return_feat=True)
    p = torch.stack(preds)
    out = {"preds": p.numpy(), "vis_e": vis_e.numpy(), "ffeat": ffeat.numpy()}
    np.savez_compressed(os.path.join(HERE, "reference_cfg4.npz"), **out)
    print("cfg4 chunk: mean |d| from init", float((p[-1] - chunk[:, None]).abs().mean()), "max", float((p[-1] - chunk[:, None]).abs().max()))
    print("wrote", os.path.join(HERE, "reference_cfg4.npz"), os.path.getsize(os.path.join(HERE, "reference_cfg4.npz")), "bytes")


# BASELINE cfg 1 on the REAL demo clip: the reference's demo_images/000100-000107.jpg decoded with PIL, the recipe of
# demo.py:21-41 (float, bilinear resize to 360 x 640, 16 x 16 query grid with an 8 px margin, model(xy, rgbs, iters=6)),
# stride 4 as demo.py:114.  The eight JPEG files (320 KB) are stored inside the fixture together with the SHA-256 of the
# decoded pixels, so that the test feeds the same bytes without a reference checkout.
DEMO_CASE = dict(B=1, H=360, W=640, N=256, stride=4, iters=6, head_scale=0.05, seed=11)
DEMO_FRAMES = list(range(100, 108))


def demo_decode(jpeg_blobs):
    """list of JPEG byte strings -> (1, S, 3, H, W) float tensor 0..255 (demo.py:134-144 reads with imageio == PIL decode)."""
    import io
    from PIL import Image
    fr = [np.array(Image.open(io.BytesIO(bytes(b))).convert("RGB")) for b in jpeg_blobs]
    return torch.from_numpy(np.stack(fr)).permute(0, 3, 1, 2).unsqueeze(0).float()


def demo_inputs(rgbs):
    """demo.py:21-36: resize to 360 x 640, 16 x 16 grid of queries (utils.basic.meshgrid2d order: y outer, x inner)."""
    import torch.nn.functional as F
    Bq, S, C, H, W = rgbs.shape
    H_, W_ = 360, 640
    rgbs = F.interpolate(rgbs.reshape(Bq * S, C, H, W), (H_, W_), mode="bilinear").reshape(Bq, S, C, H_, W_)
    N_ = 16
    gy, gx = torch.meshgrid(torch.arange(N_).float(), torch.arange(N_).float(), indexing="ij")
    gy = 8 + gy.reshape(Bq, -1) / float(N_ - 1) * (H_ - 16)
    gx = 8 + gx.reshape(Bq, -1) / float(N_ - 1) * (W_ - 16)
    return rgbs, torch.stack([gx, gy], dim=-1)


def main_demo(reference):
    import hashlib
    torch.Tensor.cuda = lambda self, *a, **k: self
    from nets.pips import Pips  # the reference, unmodified

    torch.set_num_threads(min(16, os.cpu_count() or 1))
    c = DEMO_CASE
    blobs = [open(os.path.join(reference, "demo_images", f"{i:06d}.jpg"), "rb").read() for i in DEMO_FRAMES]
    raw = demo_decode(blobs)
    rgbs, xy = demo_inputs(raw)
    sd = po.init_state_dict(seed=c["seed"], head_scale=c["head_scale"])
    model = Pips(S=8, stride=c["stride"]).eval()
    model.load_state_dict(sd, strict=True)
    with torch.no_grad():
        preds, preds2, vis_e, ffeat, _ = model(xy, rgbs, iters=c["iters"], return_feat=True)
    p = torch.stack(preds)
    out = {f"jpeg{i}": np.frombuffer(b, dtype=np.uint8) for i, b in enumerate(blobs)}
    out["pixels_sha256"] = np.array(hashlib.sha256(raw.to(torch.uint8).numpy().tobytes()).hexdigest())
    out.update({"preds": p.numpy(), "vis_e": vis_e.numpy(), "ffeat": ffeat.numpy()})
    np.savez_compressed(os.path.join(HERE, "reference_demo.npz"), **out)
    print("demo clip: mean |d| from init", float((p[-1] - xy[:, None]).abs().mean()), "max", float((p[-1] - xy[:, None]).abs().max()))
    print("wrote", os.path.join(HERE, "reference_demo.npz"), os.path.getsize(os.path.join(HERE, "reference_demo.npz")), "bytes")


# The module files of the reference's `nets` package (paths relative to the checkout, no contents): the zero-edit shim
# test rebuilds the package from empty stand-ins at these paths to check that shim/nets/pips.py shadows nets.pips only.
def main_nets_layout(reference):
    import json
    mods = sorted(os.path.relpath(os.path.join(d, f), reference).replace(os.sep, "/")
                  for d, _, files in os.walk(os.path.join(reference, "nets")) for f in files if f.endswith(".py"))
    with open(os.path.join(HERE, "reference_nets_layout.json"), "w") as f:
        json.dump(mods, f, indent=1)
    print("wrote", os.path.join(HERE, "reference_nets_layout.json"), mods)


if __name__ == "__main__":
    if "--reference" not in sys.argv[:-1]:
        sys.exit(__doc__.split("\n\n")[1])
    REFERENCE = os.path.abspath(sys.argv[sys.argv.index("--reference") + 1])
    sys.path.insert(0, REFERENCE)
    if "--cfg2" in sys.argv:
        main_cfg2()
    elif "--cfg4" in sys.argv:
        main_cfg4()
    elif "--demo" in sys.argv:
        main_demo(REFERENCE)
    elif "--nets-layout" in sys.argv:
        main_nets_layout(REFERENCE)
    else:
        main()
