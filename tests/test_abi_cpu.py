"""CPU-side checks: the C-ABI library builds, loads and exports every symbol of include/pips_b200.h;
the module mirrors the reference's state_dict; error paths do not need a GPU."""
import os
import re

import torch

from oracle import pips_oracle as po
from pips_b200 import Pips, _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_are_exported():
    hdr = open(os.path.join(ROOT, "include", "pips_b200.h")).read()
    declared = set(re.findall(r"^(?:int|size_t|const char\*)\s+(pips_\w+)\s*\(", hdr, flags=re.M))
    assert declared == set(L.EXPORTS), declared ^ set(L.EXPORTS)
    lib = L.load()
    for name in declared:
        assert hasattr(lib, name)
    macro = int(re.search(r"#define PIPS_B200_ABI_VERSION (\d+)", hdr).group(1))
    assert lib.pips_abi_version() == macro == L.ABI_VERSION == 3


def test_argument_validation_without_gpu():
    lib = L.load()
    assert lib.pips_gemm_tc(0, 0, 512, 128, 0, 0, 512, 256, 128, 256, 100, 0, 0, 0, 0, 0, 0, 0, 0) != 0
    assert b"multiple of 64" in lib.pips_last_error()
    assert lib.pips_corr_gather(None, 0, 1, 7, 1, 16, 16, 0, 0, 0, None, 0, 0, 0, 0, 576, 0) != 0
    assert lib.pips_refine_iter(None, None, None, 0, 0) != 0
    # round-2 entry points: the row-ring convolution and the statistics finalize
    assert lib.pips_conv_rows(None, None, 1, 8, 8, None, None, None, None, None) != 0 and b"null pointer" in lib.pips_last_error()
    assert lib.pips_conv_rows_chunks(192, 256) == 1 * 24 * 2 and lib.pips_conv_rows_chunks(180, 640) == 3 * 23 * 2
    assert lib.pips_conv_rows_chunks(0, 5) == 0
    assert lib.pips_inorm_finalize(None, 1, 1, 1, 64, None, None) != 0
    assert lib.pips_stem_pack(None, 0, 1, 8, 8, None, None, None) != 0


def test_state_dict_contract_matches_reference_spec():
    m = Pips(S=8, stride=4)
    spec = dict(po.state_dict_spec())
    sd = m.state_dict()
    assert list(sd) == [k for k, _ in po.state_dict_spec()]          # same names, same order
    assert all(tuple(v.shape) == spec[k] for k, v in sd.items())
    m.load_state_dict(po.init_state_dict(0), strict=True)
    assert sum(p.numel() for p in m.parameters()) == 28677713


def test_torch_modules_equal_oracle_on_cpu():
    sd = po.init_state_dict(1)
    m = Pips(S=8, stride=8).eval()
    m.load_state_dict(sd)
    x = torch.randn(3, 8, 519)
    with torch.no_grad():
        assert (m.delta_block(x) - po.mixer(sd, x).reshape(3, 8, 130)).abs().max() < 1e-6
        rgb = po.smooth_video(1, 2, 64, 96)
        inp = (2 * (rgb / 255) - 1).reshape(2, 3, 64, 96)
        assert (m.fnet(inp) - po.fnet(sd, inp, 8)).abs().max() < 1e-6


def test_edge_shapes_are_rejected_by_the_c_abi():
    """Argument validation needs no GPU: empty problems, S != 8, bad leading dimensions."""
    lib = L.load()
    assert lib.pips_update(0, 0, 0, 0, 0, 0, 0, 0, 0, 8.0, 1, 8, 1, 0) != 0
    assert b"null" in lib.pips_last_error()
    assert lib.pips_conv_tc(1, 1, 1, 16, 16, 100, 1, 1, 64, 3, 3, 1, 1, 0, 1, 0) != 0        # Cp not a multiple of 64
    assert lib.pips_conv_tc(1, 1, 1, 16, 16, 64, 1, 1, 64, 3, 3, 3, 1, 0, 1, 0) != 0         # stride 3
    assert lib.pips_tokenmix(1, 0, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0) != 0                  # zero sequences
    assert lib.pips_pyramid_build(1, 8, 4, 4, None, None, 0) != 0                            # map too small for 4 levels


def test_peer_entry_points_validate_arguments_without_gpu():
    import ctypes as C
    lib = L.load()
    assert lib.pips_peer_scatter(None, 4, 4, None, 2, 8, 0, None) != 0
    assert b"pips_peer_scatter" in lib.pips_last_error()
    one = (C.c_void_p * 1)(C.c_void_p(256))
    assert lib.pips_peer_scatter(C.c_void_p(256), 4, 4, one, 1, 6, 4, None) != 0          # block leaves the row
    assert b"outside the destination row" in lib.pips_last_error()
    assert lib.pips_peer_scatter(C.c_void_p(256), 4, 4, one, L.MAX_PEERS + 1, 8, 0, None) != 0
    assert lib.pips_peer_barrier(one, 1, 1, 1, 1000, None) != 0                            # rank outside n_peers
    assert b"bad rank" in lib.pips_last_error()
    assert lib.pips_peer_barrier(one, 0, 1, 1, 0, None) != 0                               # no timeout: could hang a device
    assert lib.pips_peer_open(None, None) != 0 and lib.pips_peer_close(None) != 0 and lib.pips_peer_free(None) != 0
    peer = L.PeerOut()
    peer.n_peers, peer.n_offset, peer.n_total = 2, 6, 8                                     # 6 + N(=4) > 8
    peer.out[0] = peer.out[1] = 256
    p = C.c_void_p(256)
    assert lib.pips_update_peer(p, p, p, p, p, p, p, p, p, 8.0, 1, 8, 4, C.byref(peer), None) != 0
    assert b"particle slice outside n_total" in lib.pips_last_error()


def test_peer_plan_layout():
    """Slab regions of one forward: disjoint, 8-byte aligned coordinate blocks, sized by words_needed."""
    from pips_b200.peer import FLAG_WORDS, PeerPlan

    class FakeSlab:
        world, rank, local, generation = 4, 2, 0x7000000000, 1
        ptrs = [0x7000000000 + r * (1 << 30) for r in range(4)]

    plan = PeerPlan(FakeSlab(), iters=6, B=4, S=8, per=257)
    assert plan.n_total == 4 * 257 and plan.n_offset == 2 * 257
    assert plan.words == PeerPlan.words_needed(4, 6, 4, 8, 257)
    assert FLAG_WORDS >= L.MAX_PEERS and plan.off_coords == FLAG_WORDS < plan.off_vis < plan.off_ffeat < plan.words
    bases = [plan.coord_bases(it) for it in range(6)]
    step = 4 * 4 * 8 * plan.n_total * 2
    for it in range(6):
        for r in range(4):
            assert bases[it][r] == FakeSlab.ptrs[r] + 4 * FLAG_WORDS + it * step and bases[it][r] % 8 == 0
    assert bases[5][0] + step == FakeSlab.ptrs[0] + 4 * plan.off_vis
    # a re-allocated slab (new generation) never shares a graph plan with the old one, even at the same address
    FakeSlab.generation = 2
    assert PeerPlan(FakeSlab(), iters=6, B=4, S=8, per=257).key != plan.key


def test_no_particles_raises_like_the_reference():
    """N = 0: the reference raises RuntimeError (F.interpolate of the empty volume, nets/pips.py:509; recorded from
    the unmodified reference by tests/golden/make_golden.py as edge/n0_error); the drop-in raises the same type."""
    import numpy as np
    import pytest
    gold = np.load(os.path.join(ROOT, "tests", "golden", "reference_outputs.npz"))
    assert str(gold["edge/n0_error"]) == "RuntimeError"
    model = Pips(S=8, stride=8).eval()
    with pytest.raises(RuntimeError):
        model(torch.zeros(2, 0, 2), po.smooth_video(2, 8, 64, 64, seed=1), iters=3)


def test_plain_c_consumer_links_and_struct_layouts_match(tmp_path):
    """examples/abi_check.c (C99, -Werror) includes the header, links the library without torch and exercises the
    validation paths; the struct sizes it prints must equal the ctypes mirrors in pips_b200/_lib.py."""
    import ctypes
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        import pytest
        pytest.skip("no gcc")
    L.load()
    exe = str(tmp_path / "abi_check")
    libdir = os.path.join(ROOT, "pips_b200", "lib")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", "abi_check.c"), "-L" + libdir, "-lpips_b200", "-Wl,-rpath," + libdir,
                    "-o", exe], check=True, capture_output=True, text=True)
    out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    assert "all checks passed" in out, out
    sizes = dict(re.findall(r"sizeof\((\w+)\)=(\d+)", out))
    assert int(sizes["pips_weights"]) == ctypes.sizeof(L.Weights)
    assert int(sizes["pips_workspace"]) == ctypes.sizeof(L.Workspace)
    assert int(sizes["pips_problem"]) == ctypes.sizeof(L.Problem)


def test_zero_edit_shim_serves_nets_pips(tmp_path):
    """shim/ before the reference on sys.path: `from nets.pips import Pips` (demo.py:9) is pips_b200.Pips, every other
    module of the reference's `nets` package still resolves to the reference checkout.  The checkout is stood in for by
    empty modules at the paths recorded from it (tests/golden/reference_nets_layout.json); its nets/pips.py fails if imported."""
    import json
    import subprocess
    import sys
    with open(os.path.join(ROOT, "tests", "golden", "reference_nets_layout.json")) as f:
        layout = json.load(f)
    assert "nets/pips.py" in layout and "nets/raft_core/util.py" in layout
    ref = tmp_path / "reference"
    for rel in layout:
        (ref / rel).parent.mkdir(parents=True, exist_ok=True)
        (ref / rel).write_text("raise ImportError('the reference nets.pips shadowed the shim')\n" if rel == "nets/pips.py" else "")
    others = [rel[:-3].replace("/", ".").removesuffix(".__init__") for rel in layout if rel != "nets/pips.py"]
    code = ("import importlib; from nets.pips import Pips; import pips_b200; assert Pips is pips_b200.Pips; "
            "m = Pips(S=8, stride=4); assert len(m.state_dict()) == 200; print('shim ok'); "
            f"assert all(importlib.import_module(n).__file__.startswith({str(ref)!r}) for n in {others!r}); "
            "print('reference nets.* still visible')")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "shim"), ROOT, str(ref)]))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "shim ok" in out.stdout and "reference nets.* still visible" in out.stdout
