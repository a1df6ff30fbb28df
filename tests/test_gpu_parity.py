"""GPU parity: the CUDA path (through the C ABI) against the oracle on the same seeded inputs and against the golden
vectors minted from the unmodified reference.  Tolerances are stated per test.  Run with `-m gpu` on a B200."""
import numpy as np
import pytest
import torch

from neo360_b200 import synth
from oracle import neo360_oracle as orc

pytestmark = pytest.mark.gpu
T = lambda a: torch.from_numpy(np.asarray(a))


@pytest.fixture(scope="module")
def cuda():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from neo360_b200 import build
    build.build()
    return torch.device("cuda:0")


def md(a, b):
    return float((a.detach().cpu().double() - b.detach().cpu().double()).abs().max())


def rays_in_sphere(n, seed):
    g = torch.Generator().manual_seed(seed)
    o = (torch.rand(n, 3, generator=g) - 0.5) * 1.1
    d = torch.randn(n, 3, generator=g)
    return o, d / d.norm(dim=-1, keepdim=True)


# ---------------- stage-level parity (bit-level or few-ulp) ----------------

def test_get_rays(cuda):
    from neo360_b200 import ops
    pose = synth.target_pose(7, 100)
    for (H, W) in ((6, 8), (48, 64), (480, 640)):
        o, vd, rd, rad = ops.get_rays(H, W, 0.8 * W, pose.to(cuda))
        ro, rvd, rrd, rrad = orc.rays_from_pose(orc.ray_directions(H, W, 0.8 * W), pose[:3, :4])
        assert md(o, ro) == 0 and md(vd, rvd) < 2e-7 and md(rd, rrd) < 2e-7 and md(rad, rrad) < 2e-7   # row-difference cancellation amplifies matmul rounding


def test_sample_rays_training_batch(cuda):
    """f3 (nerds360_ae.py:730-764): sampled-pixel rays are bit-identical to the same pixels of the whole-frame generator, match the oracle's
    build-everything-then-index restatement, and the batch dict carries the reference's keys."""
    from neo360_b200 import batches, ops
    Tn, H, W, focal = 5, 48, 64, 51.2
    poses = torch.stack([synth.target_pose(3 * k + 1, 100)[:3, :4] for k in range(Tn)])
    g = torch.Generator().manual_seed(5)
    images = torch.rand(Tn, H, W, 3, generator=g)
    pix = batches.draw_pix_inds(Tn, H, W, 500, torch.Generator().manual_seed(9))
    assert torch.equal(pix, torch.randint(0, Tn * H * W, (500,), generator=torch.Generator().manual_seed(9)))   # the reference's own draw
    pix[:4] = torch.tensor([0, W - 1, Tn * H * W - 1, (H - 1) * W])                                                # corners, last row (radii quirk)
    o, vd, rd, rad, tgt = ops.sample_rays(pix.to(cuda), H, W, focal, poses.to(cuda), images.to(cuda))
    full = [ops.get_rays(H, W, focal, p.to(cuda)) for p in poses]
    for got, k in ((o, 0), (vd, 1), (rd, 2)):
        assert torch.equal(got, torch.cat([f[k] for f in full], 0)[pix.to(cuda)])
    assert torch.equal(rad[:, 0], torch.cat([f[3] for f in full], 0)[pix.to(cuda)])
    assert torch.equal(tgt.cpu(), images.reshape(-1, 3)[pix])
    ro, rvd, rrd, rrad, rtgt = orc.sample_training_rays(pix, H, W, focal, poses, images)
    assert md(o, ro) == 0 and md(vd, rvd) < 2e-7 and md(rd, rrd) < 2e-7 and md(rad, rrad) < 2e-7 and md(tgt, rtgt) == 0
    with pytest.raises(IndexError):
        ops.sample_rays(torch.tensor([Tn * H * W], device=cuda), H, W, focal, poses.to(cuda))
    assert ops.sample_rays(torch.empty(0, dtype=torch.int64, device=cuda), H, W, focal, poses.to(cuda))[0].shape == (0, 3)
    views = batches.TargetViews(poses.to(cuda), images.to(cuda), focal)
    src = {"src_imgs": torch.zeros(3, 3, H, W, device=cuda), "src_poses": torch.zeros(3, 4, 4, device=cuda),
           "src_focal": torch.zeros(3, device=cuda), "src_c": torch.zeros(3, 2, device=cuda)}
    b = batches.train_batch(views, src, generator=torch.Generator().manual_seed(9))
    assert list(b) == ["src_imgs", "src_poses", "src_focal", "src_c", "instance_mask", "rays_o", "rays_d", "viewdirs", "target", "nocs_2d",
                       "radii", "multloss", "normals"]                                                          # nerds360_ae.py:750-764
    assert b["rays_o"].shape == (500, 3) and b["radii"].shape == (500, 1) and b["multloss"].shape == (500, 1)
    assert torch.equal(b["rays_o"][4:], o[4:]) and torch.equal(b["target"][4:], tgt[4:])


def test_sample_rays_golden(cuda):
    """Row f3 against the unmodified reference's vectors (tests/golden/train_batch_vectors.npz, oracle/make_golden_batch.py)."""
    import os
    from neo360_b200 import ops
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "train_batch_vectors.npz"))
    Tn, H, W = int(z["T"]), int(z["H"]), int(z["W"])
    images = torch.rand(Tn, H, W, 3, generator=torch.Generator().manual_seed(int(z["seed"])))
    o, vd, rd, rad, tgt = ops.sample_rays(T(z["pix_inds"]).to(cuda), H, W, float(z["focal"]), T(z["poses"]).to(cuda), images.to(cuda))
    assert md(o, T(z["rays_o"])) == 0 and md(tgt, T(z["target"])) == 0
    assert md(vd, T(z["viewdirs"])) < 2e-7 and md(rd, T(z["rays_d"])) < 2e-7 and md(rad, T(z["radii"])) < 2e-7


def test_intersect_and_coarse_sampling(cuda, golden):
    from neo360_b200 import ops
    o, d = T(golden["kat_o"]), T(golden["kat_d"])
    far = ops.intersect_sphere(o.to(cuda), d.to(cuda))
    assert md(far, T(golden["kat_far"])) <= 2.4e-7          # <= 2 ulp at ~1
    farc = T(golden["kat_far"]).to(cuda)
    near = torch.full_like(farc, 1e-4)
    t, p = ops.sample_along_rays(o.to(cuda), d.to(cuda), 4, near, farc, False, False, True)
    assert md(t, T(golden["kat_fg_t"])) == 0 and md(p, T(golden["kat_fg_p"])) == 0
    s, bp, bl = ops.sample_along_rays(o.to(cuda), d.to(cuda), 4, near, farc, False, False, False, far_uncontracted=3)
    assert md(s, T(golden["kat_bg_s"])) == 0 and md(bl, T(golden["kat_bg_l"])) == 0
    assert md(bp, T(golden["kat_bg_p"])) < 2e-6          # asin/sin/cos differ by ulps between libm and CUDA
    u = T(golden["kat_u"]).to(cuda)
    tr, _ = ops.sample_along_rays(o.to(cuda), d.to(cuda), 4, near, farc, True, False, True, u_rand=u)
    sr, _, lr = ops.sample_along_rays(o.to(cuda), d.to(cuda), 4, near, farc, True, False, False, 3, u_rand=u)
    assert md(tr, T(golden["kat_fg_t_rand"])) == 0 and md(sr, T(golden["kat_bg_s_rand"])) == 0
    assert md(lr, T(golden["kat_bg_l_rand"])) == 0
    # larger seeded case against the oracle, n_coarse = 128 (config 2)
    o, d = rays_in_sphere(4096, 3)
    far = orc.intersect_sphere(o, d)
    assert md(ops.intersect_sphere(o.to(cuda), d.to(cuda)), far) <= 4e-7
    t, p = ops.sample_along_rays(o.to(cuda), d.to(cuda), 128, None, far.to(cuda), False, False, True)
    t2, p2 = orc.sample_fg(o, d, 128, torch.full_like(far, 1e-4), far)
    assert md(t, t2) == 0 and md(p, p2) == 0
    with pytest.raises(AssertionError):                  # helper.py:271
        ops.intersect_sphere(torch.tensor([[2.0, 0, 0]], device=cuda), torch.tensor([[0.0, 1, 0]], device=cuda))


def test_volumetric_rendering(cuda, golden):
    from neo360_b200 import ops
    g = golden
    rgb, sig, d = T(g["kat_rgb"]).to(cuda), T(g["kat_sig"]).to(cuda), T(g["kat_d"]).to(cuda)
    fc = ops.volumetric_rendering(rgb, sig, T(g["kat_fg_t"]).to(cuda), d, False, True, t_far=T(g["kat_far"]).to(cuda), out_depth=True)
    for a, k in zip(fc, ("kat_fg_comp", "kat_fg_acc", "kat_fg_w", "kat_fg_lam", "kat_fg_depth")):
        assert md(a, T(g[k])) < 3e-7, k
    bc = ops.volumetric_rendering(rgb, sig, T(g["kat_bg_s"]).to(cuda), d, False, False, out_depth=True)
    for a, k in zip((bc[0], bc[1], bc[2], bc[4]), ("kat_bg_comp", "kat_bg_acc", "kat_bg_w", "kat_bg_depth")):
        assert md(a, T(g[k])) < 3e-7, k
    # config-2 length (193 samples), white background, against the oracle
    gen = torch.Generator().manual_seed(5)
    n, N = 2048, 193
    o, dd = rays_in_sphere(n, 11)
    far = orc.intersect_sphere(o, dd)
    t = torch.sort(torch.rand(n, N, generator=gen), -1).values * far
    rgb = torch.rand(n, N, 3, generator=gen)
    sig = torch.rand(n, N, 1, generator=gen) * 8
    ref = orc.composite(rgb, sig, t, dd, True, True, far)
    got = ops.volumetric_rendering(rgb.to(cuda), sig.to(cuda), t.to(cuda), dd.to(cuda), True, True, t_far=far.to(cuda), out_depth=True)
    for a, b in zip(got, ref):
        assert md(a, b) < 2e-6
    # size-independent properties: weights >= 0, sum(w) == acc, acc + lambda == 1 (up to the 1e-10 eps, quirk Q9)
    comp, acc, w, lam, _ = got
    assert float(w.min()) >= 0 and md(w.sum(-1), acc) < 1e-5 and md(acc + lam[:, 0], torch.ones(n)) < 1e-4


def test_sample_pdf(cuda, golden):
    from neo360_b200 import ops
    g = golden
    o, d, far = T(g["kat_o"]).to(cuda), T(g["kat_d"]).to(cuda), T(g["kat_far"]).to(cuda)
    # fg: t = sort(t_old U invCDF)
    t_old, w = T(g["kat_fg_t"]), T(g["kat_fg_w"])
    exp = torch.sort(torch.cat([t_old, T(g["kat_pdf_fg"])], -1), -1).values
    t, p = ops.sample_pdf(t_old.to(cuda), w.to(cuda), o, d, 6, False, True, far)
    assert md(t, exp) < 2e-7
    exp_r = torch.sort(torch.cat([t_old, T(g["kat_pdf_rand"])], -1), -1).values
    t, _ = ops.sample_pdf(t_old.to(cuda), w.to(cuda), o, d, 6, True, True, far, u_rand=T(g["kat_u6"]).to(cuda))
    assert md(t, exp_r) < 2e-7
    # bg: descending bins (quirk Q17), output flipped to descending
    s_old, wb = T(g["kat_bg_s"]), T(g["kat_bg_w"])
    exp_b = torch.flip(torch.sort(torch.cat([s_old, T(g["kat_pdf_bg"])], -1), -1).values, dims=[-1])
    s, bp, bl = ops.sample_pdf(s_old.to(cuda), wb.to(cuda), o, d, 6, False, False, far, 3.0)
    assert md(s, exp_b) < 2e-7
    # config-2 sizes vs oracle: 129 old + 64 new.  The inverse CDF is discontinuous in the bg case, so compare
    # robustly: all but a handful of samples within 1e-6, every sample inside [0,1] and sorted.
    n = 2048
    oo, dd = rays_in_sphere(n, 21)
    fr = orc.intersect_sphere(oo, dd)
    t0, _ = orc.sample_fg(oo, dd, 128, torch.full_like(fr, 1e-4), fr)
    gen = torch.Generator().manual_seed(2)
    wts = torch.rand(n, 129, generator=gen) ** 4
    wts[::7] *= 1e-9                                         # exercises the 1e-5 padding branch (helper.py:178-182)
    t_ref, _ = orc.resample_fg(oo, dd, t0, wts, 64)
    t_got, p_got = ops.sample_pdf(t0.to(cuda), wts.to(cuda), oo.to(cuda), dd.to(cuda), 64, False, True, fr.to(cuda))
    # the inverse CDF amplifies cumsum rounding by 1/pdf in low-probability bins (any two summation orders differ
    # there, e.g. torch CPU vs torch CUDA), so: >=99% of samples within 2e-6, all within one coarse bin (far/128)
    dt = (t_got.cpu() - t_ref).abs()
    assert float((dt > 2e-6).float().mean()) < 0.01 and float((dt / fr).max()) < 1.0 / 128
    assert bool((t_got[:, 1:] >= t_got[:, :-1]).all())
    s0, _, _ = orc.sample_bg(oo, dd, 128, fr)
    s_ref, bp_ref, bl_ref = orc.resample_bg(oo, dd, s0, wts, 64, fr)
    s_got, bp_got, bl_got = ops.sample_pdf(s0.to(cuda), wts.to(cuda), oo.to(cuda), dd.to(cuda), 64, False, False, fr.to(cuda), 3.0)
    # quirk Q17 makes every bg sample span the WHOLE bin range (b0 = bins[0], b1 = bins[-1]), so cumsum rounding of
    # ~1e-7 in the CDF is amplified by ~1/pdf ~ 1e2..1e3: compare at 1e-4 instead of 2e-6
    bad = ((s_got.cpu() - s_ref).abs() > 1e-4).float().mean()
    assert float(bad) < 1e-2, float(bad)
    assert bool((s_got[:, 1:] <= s_got[:, :-1]).all()) and float(s_got.min()) >= 0 and float(s_got.max()) <= 1


# ---------------- scene-dependent stages ----------------

def make_net(cuda, img_wh, plane_hw, nc, nf, seed, precisions=("fp32",), precision="fp32"):
    from neo360_b200 import NeRF_TP
    sc = synth.make_scene(img_wh, 3, plane_hw, seed)
    P = synth.make_mlp_params(seed)
    net = NeRF_TP(num_coarse_samples=nc, num_fine_samples=nf, precision=precision).eval()
    net.load_state_dict(P)
    net = net.to(cuda)
    net.set_scene(*[sc[k].to(cuda) for k in ("planes_xz", "planes_xy", "planes_yz", "latent", "src_poses", "src_focal", "src_c")],
                  sc["img_wh"], precisions=list(precisions))
    W, H = img_wh
    osc = orc.Scene(sc["planes_xz"], sc["planes_xy"], sc["planes_yz"], sc["latent"], sc["src_poses"],
                    float(sc["src_focal"][0]), float(sc["src_c"][0, 0]), float(sc["src_c"][0, 1]), W, H)
    return net, osc, P


def test_feature_lookups(cuda):
    net, osc, P = make_net(cuda, (64, 48), (24, 32), 8, 4, 0)
    g = torch.Generator().manual_seed(4)
    pts = (torch.rand(3000, 3, generator=g) - 0.5) * 3.0          # includes points that project outside -> zeros padding
    cam = orc.world2camera(pts, osc.src_poses)
    ref_w = orc.triplane_lookup(cam, osc).reshape(-1, 128)
    ref_l = orc.local_lookup(cam, osc).reshape(-1, 512)
    assert md(net.index_grid(pts.to(cuda)), ref_w) < 2e-5
    got_l = net.get_local_feats(pts.to(cuda))
    # projection through -x/(z+1e-9) amplifies ulps near z=0; compare where the reference coordinate is well conditioned
    ok = (cam[..., 2].abs() > 1e-2).reshape(-1)
    assert md(got_l.cpu()[ok], ref_l[ok]) < 5e-4


def test_field_eval_fp32_vs_oracle(cuda):
    nc = 16
    net, osc, P = make_net(cuda, (64, 48), (24, 32), nc, 8, 0)
    pose = synth.target_pose(3, 100)
    ro, vd, rd, _ = orc.rays_from_pose(orc.ray_directions(48, 64, 0.8 * 64), pose[:3, :4])
    sel = slice(1000, 1000 + 40)
    rays = {"rays_o": ro[sel].contiguous(), "rays_d": rd[sel].contiguous(), "viewdirs": vd[sel].contiguous()}
    with torch.no_grad():
        _, aux = orc.render(rays, osc, P, nc, 8, False, True, return_aux=True)
    cr = {k: v.to(cuda) for k, v in rays.items()}
    for lvl in range(2):
        for b, (tk, rk, sk) in enumerate((("fg_t", "fg_rgb", "fg_sigma"), ("bg_s", "bg_rgb", "bg_sigma"))):
            rgb, sig = net.field_eval(cr, aux[lvl]["far"].to(cuda), aux[lvl][tk].to(cuda), 2 * lvl + b, precision="fp32")
            assert md(sig, aux[lvl][sk]) < 5e-5, (lvl, b)
            assert md(rgb, aux[lvl][rk]) < 5e-5, (lvl, b)


EV = ("comp_rgb", "fg_rgb", "bg_rgb", "fg_acc", "bg_lambda", "depth")
TR = ("comp_rgb", "fg_w", "bg_w", "fg_sdist", "bg_sdist", "bg_acc")


@pytest.mark.parametrize("tag", ["tiny", "small"])
def test_end_to_end_fp32_vs_reference_vectors(cuda, golden, tag):
    """NEO_PREC_FP32 against outputs of the UNMODIFIED reference (tests/golden).  Tolerance: 2e-4 abs on every output
    (fp32 re-association through the gained MLP); bg resampling is discontinuous at CDF bracket edges (quirk Q17), so
    up to 1% of entries may exceed it, bounded by 5e-3."""
    g = golden
    W, H, hp, wp, B, nc, nf, seed, start = [int(x) for x in g[f"{tag}_cfg"]]
    net, osc, P = make_net(cuda, (W, H), (hp, wp), nc, nf, seed)
    rays = {k: T(g[f"{tag}_{k}"]).to(cuda) for k in ("rays_o", "rays_d", "viewdirs")}
    with torch.no_grad():
        ev = net(rays, False, False, 0.2, 3.0, out_depth=True)
        tr = net(rays, False, True, 0.2, 3.0, out_depth=False)
        rays_r = dict(rays)
        rays_r["_uniforms"] = [T(g[f"{tag}_u_{k}"]).to(cuda) for k in ("fg0", "bg0", "fg1", "bg1")]
        rr = net(rays_r, True, False, 0.2, 3.0, out_depth=True)
    net.check()

    def close(v, ref, name):
        diff = (v.cpu().double() - T(ref).double()).abs()
        assert float(diff.max()) < 5e-3, (name, float(diff.max()))
        assert float((diff > 2e-4).double().mean()) <= 0.01, (name, float(diff.max()))

    for lvl in range(2):
        for n_, v in zip(EV, ev[lvl]):
            close(v, g[f"{tag}_eval{lvl}_{n_}"], ("eval", lvl, n_))
        for n_, v in zip(TR, tr[lvl]):
            close(v, g[f"{tag}_train{lvl}_{n_}"], ("train", lvl, n_))
        for n_, v in zip(EV, rr[lvl]):
            close(v, g[f"{tag}_rand{lvl}_{n_}"], ("rand", lvl, n_))


def test_chunked_frame_matches_oracle_chunk_loop(cuda):
    """render_rays_test semantics: one call over a frame with chunk=C must equal the reference's Python loop over
    C-ray chunks (quirk Q1 makes the result depend on C).  48x36 frame = 1728 rays, chunk 512 (last chunk ragged)."""
    W, H, nc, nf = 48, 36, 24, 12
    net, osc, P = make_net(cuda, (W, H), (24, 32), nc, nf, 2)
    pose = synth.target_pose(11, 100)
    ro, vd, rd, _ = orc.rays_from_pose(orc.ray_directions(H, W, 0.8 * W), pose[:3, :4])
    rays = {"rays_o": ro, "rays_d": rd, "viewdirs": vd}
    with torch.no_grad():
        ref = orc.render_chunked(rays, osc, P, nc, nf, chunk=512)
        got = net.render_rays_test({k: v.to(cuda) for k, v in rays.items()}, chunk=512)
        wrong = net.render_rays_test({k: v.to(cuda) for k, v in rays.items()}, chunk=0)
    net.check()
    for k in ("rgb", "fg_rgb", "bg_rgb", "depth"):
        rk = "comp_rgb" if k == "rgb" else k
        diff = (got[k].cpu() - ref[rk]).abs()
        assert float(diff.max()) < 5e-3 and float((diff > 2e-4).float().mean()) < 0.01, (k, float(diff.max()))
    assert orc.psnr(got["rgb"].cpu(), ref["comp_rgb"]) > 60
    # walking the frame in 8x4 pixel blocks is pure scheduling: bit-identical output
    with torch.no_grad():
        blk = net.render_rays_test({k: v.to(cuda) for k, v in rays.items()}, chunk=512, img_wh=(W, H))
    for k in ("rgb", "depth"):
        assert md(blk[k], got[k]) == 0
    # sanity: ignoring the chunk size gives a measurably different image (the quirk is real and reproduced)
    assert float((wrong["rgb"].cpu() - ref["comp_rgb"]).abs().max()) > 1e-3


# ---------------- tensor-core path (NEO_PREC_TC) ----------------

def test_tc_primitives_selftest(cuda):
    """TS-mode tcgen05.mma (A in TMEM), SW128 K-major operand tiles, SS-mode MMA, TMEM loads -- against torch matmul
    on the fp16-rounded operands (exact products, fp32 accumulation: tolerance 1e-3 on O(10) sums)."""
    from neo360_b200 import _lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(0)
    X = torch.randn(128, 128, generator=g).to(cuda)
    W = torch.randn(128, 128, generator=g).to(cuda)
    Wn = torch.randn(80, 128, generator=g).to(cuda)
    o1 = torch.zeros(128, 128, device=cuda)
    o2 = torch.zeros(128, 80, device=cuda)
    o3 = torch.zeros(128, 128, device=cuda)
    o4 = torch.zeros(128, 80, device=cuda)
    L.check(lib.neo_tc_selftest(L.ptr(X), L.ptr(W), L.ptr(Wn), L.ptr(o1), L.ptr(o2), L.ptr(o3), L.ptr(o4), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    Xh, Wh, Wnh = X.half().float(), W.half().float(), Wn.half().float()
    assert md(o1, Wh @ Xh.T) < 1e-3
    assert md(o2, Xh @ Wnh.T) < 1e-3
    print("MN-major B max err", md(o3, Wh @ Xh.T), " MN-major A max err", md(o4, Xh @ Wnh.T))
    assert md(o3, Wh @ Xh.T) < 1e-3          # MN-major (point-contiguous) B operand, N=32 blocks at 64-byte offsets
    assert md(o4, Xh @ Wnh.T) < 1e-3          # MN-major A operand, M=128 as two 64-point groups


def test_tc_selftest_transpose(cuda):
    """Transpose-accumulate MMA (identity A operand in a no-swizzle K-major tile, gathered features as the SW128 K-major B
    operand): exact transposition of the fp16-rounded input.  `outa` is the descriptor reading the kernel uses."""
    from neo360_b200 import _lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(1)
    X = torch.randn(128, 128, generator=g).to(cuda)
    oa = torch.zeros(128, 128, device=cuda)
    ob = torch.zeros(128, 128, device=cuda)
    L.check(lib.neo_tc_selftest_transpose(L.ptr(X), L.ptr(oa), L.ptr(ob), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ref = X.half().float().T
    print("transpose MMA: (LBO=K stride, SBO=row-group stride) err", md(oa, ref), " swapped err", md(ob, ref))
    assert md(oa, ref) == 0.0


def test_tc_selftest_window(cuda):
    """Texel-window MMA (the bilinear lookups of the TC field kernel): one TMA box load of a 4x4x256-channel window (128B swizzle,
    zero fill outside the map) as the MN-major A operand, a sparse [64 points x 16 texels] no-swizzle K-major tap-weight tile as B.
    Exact in fp16 products / fp32 accumulation, including windows that straddle or miss the map."""
    from neo360_b200 import _lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(2)
    H, W = 6, 7
    tex = torch.randn(H * W, 256, generator=g)
    for ox, oy in ((1, 1), (-1, -2), (5, 4), (3, 2), (-4, 0), (0, 6)):
        wt = torch.rand(64, 16, generator=g) * (torch.rand(64, 16, generator=g) < 0.3)
        o0 = torch.zeros(128, 64, device=cuda)
        o3 = torch.zeros(128, 64, device=cuda)
        L.check(lib.neo_tc_selftest_window(L.ptr(tex.to(cuda)), H, W, ox, oy, L.ptr(wt.to(cuda)), L.ptr(o0), L.ptr(o3),
                                           torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        win = torch.zeros(16, 256)
        for k in range(16):
            y, x = oy + k // 4, ox + k % 4
            if 0 <= y < H and 0 <= x < W:
                win[k] = tex[y * W + x]
        ref = (wt.half().double() @ win.half().double()).T.float()          # (256, 64)
        print("window MMA at", (ox, oy), "err", md(o0, ref[:128]), md(o3, ref[128:]))
        assert md(o0, ref[:128]) < 1e-5 and md(o3, ref[128:]) < 1e-5


def test_field_eval_tc_vs_oracle(cuda):
    """TC field (fp16 operands, pre-projected features, folded head) against the oracle on identical t-values.
    Stated tolerance: |rgb| 2e-2, sigma 2e-2 + 2% (fp16 operand rounding through a 6-layer gained MLP)."""
    nc = 16
    net, osc, P = make_net(cuda, (64, 48), (24, 32), nc, 8, 0, precisions=("fp32", "tc"))
    pose = synth.target_pose(3, 100)
    ro, vd, rd, _ = orc.rays_from_pose(orc.ray_directions(48, 64, 0.8 * 64), pose[:3, :4])
    sel = slice(1000, 1000 + 75)                          # ragged: 75 rays -> 3 ray groups, last one partial
    rays = {"rays_o": ro[sel].contiguous(), "rays_d": rd[sel].contiguous(), "viewdirs": vd[sel].contiguous()}
    with torch.no_grad():
        _, aux = orc.render(rays, osc, P, nc, 8, False, True, return_aux=True)
    cr = {k: v.to(cuda) for k, v in rays.items()}
    for lvl in range(2):
        for b, (tk, rk, sk) in enumerate((("fg_t", "fg_rgb", "fg_sigma"), ("bg_s", "bg_rgb", "bg_sigma"))):
            rgb, sig = net.field_eval(cr, aux[lvl]["far"].to(cuda), aux[lvl][tk].to(cuda), 2 * lvl + b, precision="tc")
            net.check()
            ds = (sig.cpu() - aux[lvl][sk]).abs()
            assert float((ds - 0.02 * aux[lvl][sk].abs()).max()) < 2e-2, (lvl, b, float(ds.max()))
            assert md(rgb, aux[lvl][rk]) < 2e-2, (lvl, b)


@pytest.mark.parametrize("tag", ["tiny", "small"])
def test_end_to_end_tc_vs_reference_vectors(cuda, golden, tag):
    """NEO_PREC_TC against outputs of the UNMODIFIED reference.  Stated tolerance: PSNR >= 40 dB on comp_rgb,
    L-inf <= 3e-2 on rgb / acc / depth (fp16 tensor-core operands; resampling is driven by the fp16 coarse weights)."""
    g = golden
    W, H, hp, wp, B, nc, nf, seed, start = [int(x) for x in g[f"{tag}_cfg"]]
    net, osc, P = make_net(cuda, (W, H), (hp, wp), nc, nf, seed, precisions=("tc",), precision="tc")
    rays = {k: T(g[f"{tag}_{k}"]).to(cuda) for k in ("rays_o", "rays_d", "viewdirs")}
    with torch.no_grad():
        ev = net(rays, False, False, 0.2, 3.0, out_depth=True)
    net.check()
    for lvl in range(2):
        for n_, v in zip(EV, ev[lvl]):
            assert md(v, T(g[f"{tag}_eval{lvl}_{n_}"])) < 3e-2, (lvl, n_)
    assert orc.psnr(ev[1][0].cpu(), T(g[f"{tag}_eval1_comp_rgb"])) > 40


# ---------------- vanilla NeRF (row a17) ----------------

@pytest.mark.parametrize("tag", ["v_tiny", "v_cfg1"])
def test_vanilla_nerf_vs_reference_vectors(cuda, tag):
    """CUDA vanilla NeRF (fp32, reference formulation) against outputs of the UNMODIFIED reference NeRF module.
    v_cfg1 = BASELINE configs[0] (1024 rays, 64+64 samples).  Tolerance: >=99% of outputs within 2e-4, L-inf 5e-3."""
    import os
    from neo360_b200.vanilla import NeRF
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vanilla_reference_vectors.npz"))
    W, H, B, nc, nf, seed = [int(x) for x in g[f"{tag}_cfg"]]
    net = NeRF(num_coarse_samples=nc, num_fine_samples=nf).eval()
    net.load_state_dict(synth.make_vanilla_params(seed))
    net = net.to(cuda)
    rays = {k: T(g[f"{tag}_{k}"]).to(cuda) for k in ("rays_o", "rays_d", "viewdirs")}
    with torch.no_grad():
        ev = net(rays, False, True, 0.2, 3.0, debug=True)
        dbg = net.last_debug
        rays_r = dict(rays)
        rays_r["_uniforms"] = [T(g[f"{tag}_u0"]).to(cuda), T(g[f"{tag}_u1"]).to(cuda)]
        rr = net(rays_r, True, False, 0.2, 3.0)
    torch.cuda.synchronize()
    if tag == "v_tiny":      # stratified positions are bit-exact
        assert md(dbg["t"][0], T(g["v_tiny_aux0_t"])) == 0
        assert md(dbg["sigma"][0], T(g["v_tiny_aux0_sigma"])) < 1e-4 and md(dbg["rgb_s"][0], T(g["v_tiny_aux0_rgb"])) < 1e-4
    for lvl in range(2):
        for n_, a, b in zip(("rgb", "acc", "depth"), ev[lvl], rr[lvl]):
            for got, ref in ((a, g[f"{tag}_eval{lvl}_{n_}"]), (b, g[f"{tag}_rand{lvl}_{n_}"])):
                diff = (got.cpu().double() - T(ref).double()).abs()
                assert float(diff.max()) < 5e-3 and float((diff > 2e-4).double().mean()) <= 0.01, (lvl, n_, float(diff.max()))


@pytest.mark.parametrize("tag", ["v_tiny", "v_cfg1"])
def test_vanilla_nerf_tc_vs_reference_vectors(cuda, tag):
    """Vanilla NeRF with the 8 x 256 MLP layer by layer on tcgen05 (NEO_PREC_TC, fp16 weights / activations) against outputs of the
    UNMODIFIED reference module (v_cfg1 = BASELINE configs[0]).  Stated: L-inf <= 3e-2 on rgb / acc, PSNR >= 40 dB; coarse sample
    positions bit-exact."""
    import os
    from neo360_b200.vanilla import NeRF
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vanilla_reference_vectors.npz"))
    W, H, B, nc, nf, seed = [int(x) for x in g[f"{tag}_cfg"]]
    net = NeRF(num_coarse_samples=nc, num_fine_samples=nf).eval()
    net.precision = "tc"
    net.load_state_dict(synth.make_vanilla_params(seed))
    net = net.to(cuda)
    rays = {k: T(g[f"{tag}_{k}"]).to(cuda) for k in ("rays_o", "rays_d", "viewdirs")}
    with torch.no_grad():
        ev = net(rays, False, True, 0.2, 3.0, debug=True)
    torch.cuda.synchronize()
    if tag == "v_tiny":
        assert md(net.last_debug["t"][0], T(g["v_tiny_aux0_t"])) == 0
    for lvl in range(2):
        e_rgb, e_acc = md(ev[lvl][0], T(g[f"{tag}_eval{lvl}_rgb"])), md(ev[lvl][1], T(g[f"{tag}_eval{lvl}_acc"]))
        ps = orc.psnr(ev[lvl][0].cpu(), T(g[f"{tag}_eval{lvl}_rgb"]))
        print(f"vanilla tc [{tag}] level {lvl}: L-inf rgb {e_rgb:.2e} acc {e_acc:.2e} PSNR {ps:.1f} dB")
        assert e_rgb < 3e-2 and e_acc < 3e-2 and ps > 40.0, (lvl, e_rgb, e_acc, ps)


def test_tc_blocked_frame_order_is_pure_scheduling(cuda):
    """NEO_PREC_TC with NeoRays.ray_order (8x4 pixel blocks) against the identity order.  The ray order decides which 64 points
    share a job and therefore how a point's texel windows are grouped, i.e. the order of its fp32 accumulation on the tensor pipe:
    the pixels agree to accumulation rounding (stated: 1e-3 on rgb in [0,1] / depth), not bit for bit.  (Line 243 keeps the
    bit-exact check for the fp32 CUDA-core path.)"""
    W, H, nc, nf = 48, 36, 24, 12
    net, osc, P = make_net(cuda, (W, H), (24, 32), nc, nf, 2, precisions=("tc",), precision="tc")
    pose = synth.target_pose(11, 100)
    ro, vd, rd, _ = orc.rays_from_pose(orc.ray_directions(H, W, 0.8 * W), pose[:3, :4])
    rays = {"rays_o": ro.to(cuda), "rays_d": rd.to(cuda), "viewdirs": vd.to(cuda)}
    with torch.no_grad():
        a = net.render_rays_test(rays, chunk=512)
        b = net.render_rays_test(rays, chunk=512, img_wh=(W, H))
    net.check()
    for k in ("rgb", "fg_rgb", "bg_rgb", "depth"):
        assert md(a[k], b[k]) < 1e-3, k


# ---------------- Mip-NeRF 360 (row a18) ----------------

@pytest.mark.parametrize("tag", ["m_tiny", "m_small"])
def test_mip360_vs_reference_vectors(cuda, tag):
    """CUDA Mip-NeRF 360 (fp32, reference formulation, closed-form contraction Jacobian) against outputs of the UNMODIFIED
    reference MipNeRF360 module: renderings and the whole ray history of all three levels.  Tolerance 2e-4 (99%), L-inf 5e-3."""
    import os
    from neo360_b200.mip import MipNeRF360
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mip360_reference_vectors.npz"))
    W, H, B, npp, nn_, seed = [int(x) for x in g[f"{tag}_cfg"]]
    near, far = [float(x) for x in g[f"{tag}_near_far"]]
    net = MipNeRF360(num_prop_samples=npp, num_nerf_samples=nn_).eval()
    net.load_state_dict(synth.make_mip_params(seed))
    net = net.to(cuda)
    batch = {k: T(g[f"{tag}_{k}"]).to(cuda) for k in ("rays_o", "rays_d", "viewdirs", "radii")}
    with torch.no_grad():
        ren, hist = net(batch, 1.0, False, False, near, far)
        br = dict(batch)
        br["_uniforms"] = [T(g[f"{tag}_jit{i}"]).to(cuda) for i in range(3)]
        ren_r, hist_r = net(br, 0.5, True, False, near, far)
    torch.cuda.synchronize()

    def close(v, ref, name, tol=2e-4):
        diff = (v.cpu().double() - T(ref).double()).abs()
        assert float(diff.max()) < 5e-3 and float((diff > tol).double().mean()) <= 0.01, (name, float(diff.max()))

    for i in range(3):
        close(hist[i]["sdist"], g[f"{tag}_hist{i}_sdist"], (i, "sdist"), 2e-5)
        close(hist_r[i]["sdist"], g[f"{tag}_rhist{i}_sdist"], (i, "sdist rand"), 2e-5)
        for k in ("density", "rgb", "weights"):
            close(hist[i][k], g[f"{tag}_hist{i}_{k}"], (i, k))
        close(ren[i]["rgb"], g[f"{tag}_eval{i}_rgb"], (i, "rendering"))
        close(ren_r[i]["rgb"], g[f"{tag}_rand{i}_rgb"], (i, "rendering rand"))


@pytest.mark.parametrize("tag", ["m_tiny", "m_small"])
def test_mip360_tc_vs_reference_vectors(cuda, tag):
    """Mip-NeRF 360 with every dense layer on tcgen05 (NEO_PREC_TC: fp16 weights / activations, fp32 accumulate, csrc/gemm_tc.cu) against
    outputs of the UNMODIFIED reference module.  Stated: level-0 sample positions exact (no MLP upstream); renderings L-inf <= 3e-2 and
    PSNR >= 35 dB per level; fp32 CUDA path of the same weights within the same bound (it is itself within 2e-4 of the reference)."""
    import os
    from neo360_b200.mip import MipNeRF360
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mip360_reference_vectors.npz"))
    W, H, B, npp, nn_, seed = [int(x) for x in g[f"{tag}_cfg"]]
    near, far = [float(x) for x in g[f"{tag}_near_far"]]
    net = MipNeRF360(num_prop_samples=npp, num_nerf_samples=nn_, precision="tc").eval()
    net.load_state_dict(synth.make_mip_params(seed))
    net = net.to(cuda)
    batch = {k: T(g[f"{tag}_{k}"]).to(cuda) for k in ("rays_o", "rays_d", "viewdirs", "radii")}
    with torch.no_grad():
        ren, hist = net(batch, 1.0, False, False, near, far)
    torch.cuda.synchronize()
    assert md(hist[0]["sdist"], T(g[f"{tag}_hist0_sdist"])) < 2e-5
    for i in range(3):
        err = md(ren[i]["rgb"], T(g[f"{tag}_eval{i}_rgb"]))
        ps = orc.psnr(ren[i]["rgb"].cpu(), T(g[f"{tag}_eval{i}_rgb"]))
        print(f"mip tc [{tag}] level {i}: rendering L-inf {err:.2e}, PSNR {ps:.1f} dB")
        assert err < 3e-2 and ps > 35.0, (i, err, ps)


# ---------------- edge cases of the NeO-360 path ----------------

def _frame_rays(W, H, view=3):
    pose = synth.target_pose(view, 100)
    ro, vd, rd, _ = orc.rays_from_pose(orc.ray_directions(H, W, 0.8 * W), pose[:3, :4])
    return {"rays_o": ro, "rays_d": rd, "viewdirs": vd}


@pytest.mark.parametrize("nv", [1, 2, 4, 8])
def test_other_source_view_counts(cuda, nv):
    """NV != 3 source views (NeRF_TP(num_src_views=...), model.py:173): fp32 within 2e-4 of the oracle, TC within 3e-2.  NV = 8 is the
    TC kernel's kMaxViews; the fp32 path is built for 1..4 views and refuses more."""
    from neo360_b200 import NeRF_TP
    W, H, nc, nf = 64, 48, 16, 8
    sc = synth.make_scene((W, H), nv, (24, 32), 5)
    P = synth.make_mlp_params(5)
    osc = orc.Scene(sc["planes_xz"], sc["planes_xy"], sc["planes_yz"], sc["latent"], sc["src_poses"],
                    float(sc["src_focal"][0]), float(sc["src_c"][0, 0]), float(sc["src_c"][0, 1]), W, H)
    rays = {k: v[700:700 + 50].contiguous() for k, v in _frame_rays(W, H).items()}
    with torch.no_grad():
        ref = orc.render(rays, osc, P, nc, nf, False, True)[1]
    net = NeRF_TP(num_coarse_samples=nc, num_fine_samples=nf, num_src_views=nv, precision="fp32").eval()
    net.load_state_dict(P)
    net = net.to(cuda)
    net.set_scene(*[sc[k].to(cuda) for k in ("planes_xz", "planes_xy", "planes_yz", "latent", "src_poses", "src_focal", "src_c")],
                  sc["img_wh"], precisions=["fp32", "tc"])
    cr = {k: v.to(cuda) for k, v in rays.items()}
    for prec, tol in (("fp32", 3e-4), ("tc", 3e-2)):
        net.precision = prec
        if prec == "fp32" and nv > 4:
            with pytest.raises(RuntimeError, match="1..4 source views"), torch.no_grad():
                net(cr, False, False, None, None, out_depth=True)
            continue
        with torch.no_grad():
            got = net(cr, False, False, None, None, out_depth=True)[1]
        net.check()
        assert md(got[0], ref[0]) < tol and md(got[5], ref[5]) < tol, (prec, md(got[0], ref[0]))


def test_reference_default_sample_counts_and_ragged_sizes(cuda):
    """NeRF_TP defaults 128 + 256 samples (model.py:169-171 => 129 / 385 points) on 33 rays (one full TC ray group + one ray),
    and a single ray; fp32 vs oracle 3e-4, TC vs fp32 3e-2."""
    net, osc, P = make_net(cuda, (64, 48), (24, 32), 128, 256, 3, precisions=("fp32", "tc"))
    for n in (33, 1):
        rays = {k: v[1500:1500 + n].contiguous() for k, v in _frame_rays(64, 48).items()}
        with torch.no_grad():
            ref = orc.render(rays, osc, P, 128, 256, False, True)[1]
        cr = {k: v.to(cuda) for k, v in rays.items()}
        res = {}
        for prec in ("fp32", "tc"):
            net.precision = prec
            with torch.no_grad():
                res[prec] = net(cr, False, False, None, None, out_depth=True)[1]
            net.check()
        assert md(res["fp32"][0], ref[0]) < 3e-4, n
        assert md(res["tc"][0], res["fp32"][0].cpu()) < 3e-2, n


def test_ray_missing_the_sphere_is_reported(cuda):
    """The reference asserts (helper.py:271); here the error is deferred to NeRF_TP.check()."""
    net, osc, P = make_net(cuda, (64, 48), (24, 32), 8, 4, 0)
    rays = {"rays_o": torch.tensor([[2.0, 0.0, 0.0]], device=cuda), "rays_d": torch.tensor([[0.0, 1.0, 0.0]], device=cuda),
            "viewdirs": torch.tensor([[0.0, 1.0, 0.0]], device=cuda)}
    with torch.no_grad():
        net(rays, False, False, None, None, out_depth=True)
    with pytest.raises(RuntimeError, match="unit sphere"):
        net.check()
    net.check()      # flag is cleared after being reported


def test_tc_randomized_and_train_tuple(cuda, golden):
    """TC path with the reference's injected uniforms and the train-mode tuple layout (weights / sdist), vs reference vectors."""
    g = golden
    tag = "small"
    W, H, hp, wp, B, nc, nf, seed, start = [int(x) for x in g[f"{tag}_cfg"]]
    net, osc, P = make_net(cuda, (W, H), (hp, wp), nc, nf, seed, precisions=("tc",), precision="tc")
    rays = {k: T(g[f"{tag}_{k}"]).to(cuda) for k in ("rays_o", "rays_d", "viewdirs")}
    rays_r = dict(rays)
    rays_r["_uniforms"] = [T(g[f"{tag}_u_{k}"]).to(cuda) for k in ("fg0", "bg0", "fg1", "bg1")]
    with torch.no_grad():
        rr = net(rays_r, True, False, None, None, out_depth=True)
        tr = net(rays, False, True, None, None, out_depth=False)
    net.check()
    assert md(rr[1][0], T(g[f"{tag}_rand1_comp_rgb"])) < 3e-2 and md(rr[0][0], T(g[f"{tag}_rand0_comp_rgb"])) < 3e-2
    assert tr[1][1].shape == (B, nc + 1 + nf) and md(tr[0][3], T(g[f"{tag}_train0_fg_sdist"])) < 1e-6     # coarse sdist is exact
    assert md(tr[0][1], T(g[f"{tag}_train0_fg_w"])) < 3e-2 and md(tr[1][0], T(g[f"{tag}_train1_comp_rgb"])) < 3e-2


# ---------------- BASELINE.json full size (configs[1]: 640x480, 128+64 samples, 3 source views) ----------------

def test_full_size_frame_properties(cuda):
    """Whole-frame companion of test_headline_config_vs_oracle (which compares whole chunks of this frame with the oracle): at the
    benchmark's full size the oracle takes ~1 h per frame, so the rest of the frame is covered by size-independent properties:
    (1) idempotence: two renders of the same frame are bit-identical (no race in the persistent tensor-core kernel; texel windows
        are accumulated in a fixed order);
    (2) the 8x4-pixel-block schedule is pure scheduling: a 16 384-ray prefix rendered in row-major order agrees up to the fp32
        accumulation order of each point's texel windows (stated: 1e-3);
    (3) the tensor-core path agrees with the reference-formulation fp32 CUDA path (itself within 2e-4 of the reference vectors
        at the small sizes) on those rays: L-inf <= 3e-2 on rgb and acc, PSNR >= 40 dB;
    (4) range / compositing invariants: rgb in [-1e-3, 1+1e-3]-ish after compositing, 0 <= acc <= 1 + 1e-5, depth >= 0."""
    import bench
    from neo360_b200 import NeRF_TP
    sc, P = bench.build_scene_cpu()
    W, H = bench.IMG_W, bench.IMG_H
    net = NeRF_TP(num_coarse_samples=bench.N_COARSE, num_fine_samples=bench.N_FINE, num_src_views=bench.NV, precision="tc").eval()
    net.load_state_dict(P)
    net = net.to(cuda)
    net.set_scene(*[sc[k].to(cuda) for k in ("planes_xz", "planes_xy", "planes_yz", "latent", "src_poses", "src_focal", "src_c")],
                  sc["img_wh"], precisions=("tc", "fp32"))
    o, d = bench.frame_rays_cpu(7)
    rays = {"rays_o": o.to(cuda), "rays_d": d.to(cuda), "viewdirs": d.to(cuda)}
    with torch.no_grad():
        a = net.render_rays_test(rays, chunk=bench.CHUNK, img_wh=(W, H))
        b = net.render_rays_test(rays, chunk=bench.CHUNK, img_wh=(W, H))
        n = 16384                                         # whole chunks, so quirk Q1's conditioning rays are the same
        sub = {k: v[:n].contiguous() for k, v in rays.items()}
        c = net.render_rays_test(sub, chunk=bench.CHUNK)
        net.precision = "fp32"
        f = net.render_rays_test(sub, chunk=bench.CHUNK)
        net.precision = "tc"
    net.check()
    for k in ("rgb", "fg_rgb", "bg_rgb", "depth", "fg_acc"):
        assert md(a[k], b[k]) == 0, ("not idempotent", k)
        assert md(a[k][:n], c[k]) < 1e-3, ("block order changed the result", k)
    assert a["rgb"].shape == (W * H, 3) and torch.isfinite(a["rgb"]).all() and torch.isfinite(a["depth"]).all()
    assert float(a["rgb"].min()) >= -2e-3 and float(a["rgb"].max()) <= 1.0 + 2e-3
    assert float(a["fg_acc"].min()) >= 0.0 and float(a["fg_acc"].max()) <= 1.0 + 1e-5
    assert float(a["depth"].min()) >= 0.0
    err = md(c["rgb"], f["rgb"])
    mse = float(((c["rgb"] - f["rgb"]).double() ** 2).mean())
    psnr = -10.0 * np.log10(max(mse, 1e-30))
    print(f"full-size tc vs fp32 (16384 rays): rgb L-inf {err:.2e}, PSNR {psnr:.1f} dB, acc L-inf {md(c['fg_acc'], f['fg_acc']):.2e}")
    assert err <= 3e-2 and psnr >= 40.0
    assert md(c["fg_acc"], f["fg_acc"]) <= 3e-2


def test_headline_config_vs_oracle(cuda):
    """BASELINE.json's metric config itself (640x480 frame, 128+64 samples, NV=3, chunk=1024; the bench scene): two whole
    1024-ray chunks of the frame -- one through the image centre, one on the top rows where many lookups leave the source
    images -- rendered through `render_rays_test(chunk=1024)` with NEO_PREC_TC and NEO_PREC_FP32 and compared with the oracle's
    chunk loop on the same rays (models/neo360/model.py:861-907, models/interface.py:53-61).
    Stated tolerances: fp32: L-inf 5e-4 (rgb, acc), 5e-3 depth (CDF-bracket flips), PSNR >= 70 dB;
    TC (fp16 operands, fp32 accumulate): L-inf 1e-2 on rgb / acc, 2e-2 on depth, PSNR >= 45 dB."""
    import bench
    from neo360_b200 import NeRF_TP
    sc, P = bench.build_scene_cpu()
    W, H = bench.IMG_W, bench.IMG_H
    net = NeRF_TP(num_coarse_samples=bench.N_COARSE, num_fine_samples=bench.N_FINE, num_src_views=bench.NV, precision="tc").eval()
    net.load_state_dict(P)
    net = net.to(cuda)
    net.set_scene(*[sc[k].to(cuda) for k in ("planes_xz", "planes_xy", "planes_yz", "latent", "src_poses", "src_focal", "src_c")],
                  sc["img_wh"], precisions=("tc", "fp32"))
    osc = orc.Scene(sc["planes_xz"], sc["planes_xy"], sc["planes_yz"], sc["latent"], sc["src_poses"],
                    float(sc["src_focal"][0]), float(sc["src_c"][0, 0]), float(sc["src_c"][0, 1]), W, H)
    o, d = bench.frame_rays_cpu(0)
    torch.set_num_threads(min(32, torch.get_num_threads()))
    for start in ((H // 2) * W, 3 * W):
        rays = {"rays_o": o[start:start + bench.CHUNK].contiguous(), "rays_d": d[start:start + bench.CHUNK].contiguous(),
                "viewdirs": d[start:start + bench.CHUNK].contiguous()}
        with torch.no_grad():
            ref = orc.render_chunked(rays, osc, P, bench.N_COARSE, bench.N_FINE, chunk=bench.CHUNK, lookup_impl="aten")
            cr = {k: v.to(cuda) for k, v in rays.items()}
            for prec, (tol_c, tol_d, db) in (("fp32", (5e-4, 5e-3, 70.0)), ("tc", (1e-2, 2e-2, 45.0))):
                net.precision = prec
                got = net.render_rays_test(cr, chunk=bench.CHUNK)
                net.check()
                e_rgb, e_acc, e_dep = md(got["rgb"], ref["comp_rgb"]), md(got["fg_acc"], ref["fg_acc"]), md(got["depth"], ref["depth"])
                ps = orc.psnr(got["rgb"].cpu(), ref["comp_rgb"])
                print(f"headline chunk @{start} [{prec}]: Linf rgb {e_rgb:.2e} acc {e_acc:.2e} depth {e_dep:.2e} PSNR {ps:.1f} dB")
                assert e_rgb < tol_c and e_acc < tol_c and e_dep < tol_d and ps > db, (prec, start, e_rgb, e_acc, e_dep, ps)


def test_output_side_psnr_and_frames(cuda, tmp_path):
    """SURVEY.md 8(f4): PSNR reduced by the library's CUDA kernel equals LitModel.psnr_each (models/interface.py:53-61, oracle.psnr) to
    1e-4 dB including out-of-range pixels; gather_images at world 1 reshapes ray rows into frames; the writers produce files."""
    from neo360_b200 import output
    g = torch.Generator().manual_seed(5)
    a = torch.rand(48 * 64, 3, generator=g) * 1.2 - 0.1
    b = torch.rand(48 * 64, 3, generator=g)
    assert abs(output.psnr(a.to(cuda), b.to(cuda)) - orc.psnr(a, b)) < 1e-4
    assert output.psnr(b.to(cuda), b.to(cuda)) == float("inf")
    frames = output.gather_images(a.to(cuda), [(48, 64)], 1, 1024)
    assert frames[0].shape == (48, 64, 3) and md(frames[0].reshape(-1, 3), a) == 0
    paths = output.store_image(str(tmp_path), frames, "rgb") + output.store_depth_raw(str(tmp_path), [a[:, 0].reshape(48, 64)], "depth")
    import os
    assert all(os.path.getsize(p) > 0 for p in paths)


@pytest.mark.parametrize("M,N,K,relu", [(1000, 1024, 512, 1), (257, 256, 1536, 1), (4096, 128, 320, 1), (130, 64, 64, 0), (70000, 1024, 1024, 1),
                                          (20001, 256, 128, 0), (19000, 512, 1536, 1), (40000, 256, 256, 1), (19000, 256, 64, 1),
                                          (1, 64, 64, 0), (100, 128, 128, 1), (127, 256, 512, 0)])
def test_tc_dense_vs_torch(cuda, M, N, K, relu):
    """The tensor-core dense layer of the wide MLPs (csrc/gemm_tc.cu: TMA tile loads + tcgen05, fp16 operands, fp32 accumulate) against a
    plain PyTorch fp32 reference of the same op on the fp16-rounded operands; ragged M, M below one 128-row tile (the scene projection
    of maps with fewer than 128 texels; these also run with a NULL bias), every N tile width (64/128/256), K up to 1536;
    (70000,1024,1024) and (19000,512,1536) have a 256 x 256 tile for every SM pair and run the cta_group::2 kernel (gemm_f16_pair_kernel);
    the N = 256, K <= 256 shapes with a row tile for every SM run the weight-stationary kernel (gemm_f16_ws_kernel).
    Stated: |err| <= 2e-3 * max|ref| (fp32 accumulation order + the fp16 rounding of the output)."""
    from neo360_b200 import _lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g).to(cuda)
    W = (torch.randn(N, K, generator=g) / K ** 0.5).to(cuda)
    b = torch.randn(N, generator=g).to(cuda)
    out = torch.empty(M, N, device=cuda)
    L.check(lib.neo_tc_dense(L.ptr(A), L.ptr(W), L.ptr(b), M, N, K, relu, L.ptr(out), torch.cuda.current_stream().cuda_stream))
    ref = A.half().float() @ W.half().float().T + b
    if relu:
        ref = torch.relu(ref)
    err = float((out - ref).abs().max())
    print(f"tc dense {M}x{N}x{K}: max err {err:.3e}, max ref {float(ref.abs().max()):.3f}")
    assert err <= 2e-3 * float(ref.abs().max())
    if M < 128:
        out.fill_(float("nan"))
        L.check(lib.neo_tc_dense(L.ptr(A), L.ptr(W), None, M, N, K, relu, L.ptr(out), torch.cuda.current_stream().cuda_stream))
        ref = A.half().float() @ W.half().float().T
        ref = torch.relu(ref) if relu else ref
        assert float((out - ref).abs().max()) <= 2e-3 * float(ref.abs().max())


def test_scene_cache_is_keyed_by_identity_and_parameter_version(cuda):
    """ADVICE round 1: (1) a new scene whose tensors the caching allocator placed at the SAME addresses as the freed previous scene must
    not be rendered with the previous scene's packed maps; (2) a parameter update after the first render must be picked up (the scene
    packs the weights).  Both against the oracle (fp32 path, 2e-4)."""
    from neo360_b200 import NeRF_TP
    W, H, nc, nf = 48, 36, 12, 6
    P = synth.make_mlp_params(3)
    net = NeRF_TP(num_coarse_samples=nc, num_fine_samples=nf, precision="fp32").eval()
    net.load_state_dict(P)
    net = net.to(cuda)
    rays = {k: v[300:300 + 40].contiguous() for k, v in _frame_rays(W, H).items()}
    cr = {k: v.to(cuda) for k, v in rays.items()}
    ptrs = []
    for seed in (11, 12):
        sc = synth.make_scene((W, H), 3, (18, 24), seed)
        batch = dict(cr)
        batch.update({k: sc[k].to(cuda) for k in ("planes_xz", "planes_xy", "planes_yz", "latent", "src_poses", "src_focal", "src_c")})
        batch["src_imgs"] = torch.zeros(3, 3, H, W, device=cuda)
        ptrs.append(batch["latent"].data_ptr())
        osc = orc.Scene(sc["planes_xz"], sc["planes_xy"], sc["planes_yz"], sc["latent"], sc["src_poses"],
                        float(sc["src_focal"][0]), float(sc["src_c"][0, 0]), float(sc["src_c"][0, 1]), W, H)
        with torch.no_grad():
            got = net(batch, False, False, None, None, out_depth=True)[1]
            ref = orc.render(rays, osc, P, nc, nf, False, True)[1]
        net.check()
        assert md(got[0], ref[0]) < 2e-4, (seed, md(got[0], ref[0]))
        del batch, sc                                        # free the scene tensors: the next scene reuses the blocks
        torch.cuda.synchronize()
    print("latent addresses of the two scenes:", ptrs, "(equal = the allocator reused the block)")
    # (2) in-place parameter update: the packed weights must be rebuilt
    sc = synth.make_scene((W, H), 3, (18, 24), 13)
    net.set_scene(*[sc[k].to(cuda) for k in ("planes_xz", "planes_xy", "planes_yz", "latent", "src_poses", "src_focal", "src_c")], sc["img_wh"])
    osc = orc.Scene(sc["planes_xz"], sc["planes_xy"], sc["planes_yz"], sc["latent"], sc["src_poses"],
                    float(sc["src_focal"][0]), float(sc["src_c"][0, 0]), float(sc["src_c"][0, 1]), W, H)
    with torch.no_grad():
        a = net(cr, False, False, None, None, out_depth=True)[1][0]
        P2 = {k: v.clone() for k, v in synth.make_mlp_params(4).items()}
        net.load_state_dict(P2)                              # copies in place: same storages, new versions
        b = net(cr, False, False, None, None, out_depth=True)[1][0]
        ref2 = orc.render(rays, osc, P2, nc, nf, False, True)[1][0]
    net.check()
    assert md(a, b) > 1e-3 and md(b, ref2) < 2e-4, (md(a, b), md(b, ref2))


def test_scene_block_pool_recycles_without_stale_data(cuda):
    """Scene changes recycle the device blocks of the destroyed scene (neo_scene_free -> pool -> neo_scene_create).  A recycled block
    holds the PREVIOUS scene's packed maps: every scene must still render its own data (tc and fp32 against the oracle), and
    `release_cached` must hand the blocks back."""
    import neo360_b200
    from neo360_b200 import NeRF_TP
    W, H, nc, nf = 64, 48, 12, 6
    P = synth.make_mlp_params(5)
    rays = {k: v[500:500 + 64].contiguous() for k, v in _frame_rays(W, H).items()}
    cr = {k: v.to(cuda) for k, v in rays.items()}
    for prec, tol in (("tc", 3e-2), ("fp32", 2e-4)):
        net = NeRF_TP(num_coarse_samples=nc, num_fine_samples=nf, precision=prec).eval()
        net.load_state_dict(P)
        net = net.to(cuda)
        sizes = []
        for seed in (21, 22, 23):
            sc = synth.make_scene((W, H), 3, (24, 32), seed)
            net.set_scene(*[sc[k].to(cuda) for k in ("planes_xz", "planes_xy", "planes_yz", "latent", "src_poses", "src_focal", "src_c")],
                          sc["img_wh"])                       # destroys the previous scene: same shapes, so its blocks are reused
            sizes.append(net._scene.nbytes)
            osc = orc.Scene(sc["planes_xz"], sc["planes_xy"], sc["planes_yz"], sc["latent"], sc["src_poses"],
                            float(sc["src_focal"][0]), float(sc["src_c"][0, 0]), float(sc["src_c"][0, 1]), W, H)
            with torch.no_grad():
                got = net(cr, False, False, None, None, out_depth=True)[1]
                ref = orc.render(rays, osc, P, nc, nf, False, True)[1]
            net.check()
            assert md(got[0], ref[0]) < tol, (prec, seed, md(got[0], ref[0]))
        assert sizes[0] == sizes[1] == sizes[2]
        del net
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    neo360_b200.release_cached()
    assert torch.cuda.mem_get_info()[0] >= free0
