"""CPU: the C-ABI shared library loads and exports every symbol include/neo360_b200.h declares;
host-side argument validation that needs no GPU."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from neo360_b200 import build, _lib
    build.build()
    return _lib.load()


def test_header_symbols_all_exported(lib):
    from neo360_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "neo360_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(neo_[a-z_0-9]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SYMBOLS), (declared ^ set(_lib.SYMBOLS))
    for name in declared:
        assert hasattr(lib, name), name


def test_version_and_error_string(lib):
    assert b"sm_100a" in lib.neo_version()
    assert isinstance(lib.neo_last_error(), bytes)


def test_argument_validation_without_gpu(lib):
    from neo360_b200 import _lib as L
    cfg = L.NeoCfg()
    cfg.n_coarse, cfg.n_fine, cfg.precision = 128, 64, 0
    assert lib.neo_render_workspace_bytes(1024, C.byref(cfg)) > 1024 * (129 + 193) * 4
    cfg.n_coarse = 1
    assert lib.neo_render_workspace_bytes(1024, C.byref(cfg)) == 0
    assert b"n_coarse" in lib.neo_last_error()
    assert lib.neo_render_fwd(None, None, C.byref(cfg), None, None, 0, None) == -1
    assert lib.neo_field_eval(None, None, None, None, 8, 0, 0, None, None, None) == -1


@pytest.mark.parametrize("in_ch,ke", [(3, 64), (4, 96)])
def test_tc_encoding_column_layout_is_a_permutation(lib, in_ch, ke):
    """The TC kernel orders the positional-encoding columns per coordinate (x, sin 2^k x, cos 2^k x) so that the double-angle
    recurrence applies; the weight image is permuted with the same table.  It must cover every reference column
    (helper.py:121-125 order) exactly once, carry exactly one constant-one (bias) column and only zero padding otherwise."""
    cols = [lib.neo_tc_enc_column(in_ch, c) for c in range(ke)]
    ref = sorted(c for c in cols if c >= 0)
    assert ref == list(range(21 * in_ch))
    assert cols.count(-1) == 1 and cols.count(-2) == ke - 21 * in_ch - 1
    # per-coordinate grouping: column of x_c, then its 10 sines (levels ascending), then its 10 cosines
    stride = 21 if in_ch == 3 else 24
    for cc in range(in_ch):
        base = cc * stride
        assert cols[base] == cc
        assert cols[base + 1:base + 11] == [in_ch + k * in_ch + cc for k in range(10)]
        assert cols[base + 11:base + 21] == [in_ch + 10 * in_ch + k * in_ch + cc for k in range(10)]
    assert lib.neo_tc_enc_column(5, 0) == -3 and lib.neo_tc_enc_column(3, 64) == -3


def test_struct_layout_matches_header():
    """sizeof of the ctypes mirrors == what a C compiler lays out for the header (guards silent ABI drift)."""
    import subprocess, tempfile
    from neo360_b200 import _lib as L
    src = '#include <stdio.h>\n#include "neo360_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n", sizeof(NeoMLPParams), sizeof(NeoSceneDesc), sizeof(NeoRays), sizeof(NeoCfg), sizeof(NeoOut));return 0;}\n'
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "s.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(td, "s.c"), "-o", os.path.join(td, "s")])
        sizes = [int(x) for x in subprocess.check_output([os.path.join(td, "s")]).split()]
    assert sizes == [C.sizeof(L.NeoMLPParams), C.sizeof(L.NeoSceneDesc), C.sizeof(L.NeoRays), C.sizeof(L.NeoCfg), C.sizeof(L.NeoOut)]


def test_renderer_refuses_cpu_tensors():
    import torch
    from neo360_b200 import NeRF_TP, synth
    net = NeRF_TP(num_coarse_samples=8, num_fine_samples=4, precision="fp32").eval()
    sc = synth.make_scene((32, 24), 3, (12, 16), 0)
    with pytest.raises(RuntimeError, match="CUDA"):
        net.set_scene(sc["planes_xz"], sc["planes_xy"], sc["planes_yz"], sc["latent"], sc["src_poses"], sc["src_focal"],
                      sc["src_c"], sc["img_wh"])


@pytest.mark.parametrize("wh", [(640, 480), (48, 36), (37, 23)])
def test_blocked_frame_order_is_a_block_permutation(wh):
    """Host logic of the 8x4-pixel-block ray schedule (renderer._blocked_order): a permutation of the frame's pixels; when the frame
    is a multiple of 8x4, every run of 32 consecutive slots is exactly one 8x4 pixel block in row-major order inside the block."""
    import torch
    from neo360_b200 import NeRF_TP
    W, H = wh
    net = NeRF_TP(num_coarse_samples=8, num_fine_samples=4, precision="tc").eval()
    order = net._blocked_order(W * H, (W, H), torch.device("cpu")).long()
    assert order.dtype == torch.int64 and order.numel() == W * H
    assert torch.equal(torch.sort(order).values, torch.arange(W * H))
    if W % 8 == 0 and H % 4 == 0:
        blk = order.view(-1, 32)
        y, x = blk // W, blk % W
        assert torch.equal(y - y[:, :1], torch.arange(32).div(8, rounding_mode="floor").expand_as(y))
        assert torch.equal(x - x[:, :1], (torch.arange(32) % 8).expand_as(x))
        assert bool((x[:, 0] % 8 == 0).all()) and bool((y[:, 0] % 4 == 0).all())


@pytest.mark.parametrize("nv,hw,code", [(9, (24, 32), -5), (3, (1, 32), -1), (3, (32, 1), -1)])
def test_scene_create_refusals_without_gpu(lib, nv, hw, code):
    """neo_scene_create refuses more source views than the TC kernel's kMaxViews = 8 (NEO_ERR_UNSUPPORTED) and a 1 x k feature map
    (NEO_ERR_INVALID: grid_sample's align_corners scaling divides by size - 1) before it touches the device."""
    from neo360_b200 import _lib as L
    d = L.NeoSceneDesc()
    d.nv, d.world_ch, d.local_ch = nv, 128, 512
    d.plane_h, d.plane_w = hw
    d.lat_h, d.lat_w = 24, 32
    d.img_w, d.img_h = 64, 48
    mlps = (L.NeoMLPParams * 4)()
    h = C.c_void_p()
    assert lib.neo_scene_create(C.byref(d), mlps, 3, C.byref(h), None) == code
    assert not h.value
    assert (b"views" if nv > 8 else b"2x2") in lib.neo_last_error()
