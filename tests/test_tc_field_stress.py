"""The tensor-core field kernel (NEO_PREC_TC, csrc/field_tc.cu) against a model of its own fp16 arithmetic
(oracle/tc_field_model.py), on inputs that reach its window-ring, padding and edge paths.

The other TC tests compare the kernel with the fp32 reference formulation, so their bounds have to absorb fp16 operand rounding
(~1e-3 here, up to 3e-2 allowed).  The model rounds where the kernel rounds, which leaves only fp32 accumulation order and fast-math
geometry between the two: TC_RGB_BOUND / TC_SIGMA_BOUND below are set from the gap measured on a B200 (DESIGN.md section 2).

CPU tests (unmarked): the model is an exact re-association of the oracle when nothing is rounded, and each of a list of plausible
kernel bugs, injected into the model, moves the outputs by at least 3x the TC bound.  GPU tests (marked): scenarios A-G."""
import ctypes as C
from dataclasses import dataclass
from typing import Optional

import pytest
import torch

from neo360_b200 import synth
from oracle import neo360_oracle as orc
from oracle import tc_field_model as tm

# TC kernel vs model: |rgb| <= TC_RGB_BOUND, |sigma| <= TC_SIGMA_BOUND * (1 + sigma).  Measured worst over scenarios A-G on a B200:
# rgb 2.6e-3, sigma 8.2e-4 (DESIGN.md section 2).
TC_RGB_BOUND = 5e-3
TC_SIGMA_BOUND = 2e-3
# fp32 CUDA path vs the fp64 oracle: the bound of test_field_eval_fp32_vs_oracle; twice that for B, whose 640x480 source cameras
# (focal 512 px) turn the fp32 rounding of a point into ~1e-4 texel of the 240x320 latent
FP32_BOUND = 5e-5
TAIL = 1024                        # floats of NaN past each output (4 KB): the kernel must not write there


# ---------------- stress inputs ----------------

@dataclass
class Case:
    name: str
    img_wh: tuple
    nv: int
    plane_hw: tuple
    o: torch.Tensor
    d: torch.Tensor
    t_fg: torch.Tensor
    t_bg: torch.Tensor
    chunk: int = 0
    mlps: tuple = (0, 1)
    order: Optional[torch.Tensor] = None
    seed: int = 0

    @property
    def far(self):
        return orc.intersect_sphere(self.o, self.d)[:, 0]

    def t(self, mi):
        return self.t_bg if mi & 1 else self.t_fg


_scenes = {}


def scene(img_wh, nv, plane_hw, seed=0):
    key = (img_wh, nv, plane_hw, seed)
    if key not in _scenes:
        s = synth.make_scene(img_wh, nv, plane_hw, seed)
        _scenes[key] = (s, orc.Scene(s["planes_xz"], s["planes_xy"], s["planes_yz"], s["latent"], s["src_poses"],
                                     float(s["src_focal"][0]), float(s["src_c"][0, 0]), float(s["src_c"][0, 1]), *img_wh))
    return _scenes[key]


def scattered_rays(n, seed):
    g = torch.Generator().manual_seed(seed)
    o = (torch.rand(n, 3, generator=g) - 0.5) * 1.1
    d = torch.randn(n, 3, generator=g)
    return o, d / d.norm(dim=-1, keepdim=True)


def frame_rays(W, H, view=3):
    pose = synth.target_pose(view, 100)
    ro, vd, rd, _ = orc.rays_from_pose(orc.ray_directions(H, W, 0.8 * W), pose[:3, :4])
    return ro, rd


def sample_t(o, d, N, seed):
    """fg: sorted t in (0, far); bg: inverse radii s in (0, 1), descending like the renderer's."""
    g = torch.Generator().manual_seed(seed)
    far = orc.intersect_sphere(o, d)
    t = torch.sort(torch.rand(o.shape[0], N, generator=g), -1).values * far
    s = torch.sort(torch.rand(o.shape[0], N, generator=g), -1, descending=True).values
    return t, s


def rays_through(p, t0=0.02, step=0.05, N=4):
    """One ray per point p (k, 3) (world, inside the sphere) that passes through it at sample 0 (t = t0), heading for the origin."""
    d = -p / p.norm(dim=-1, keepdim=True).clamp_min(1e-6)
    o = p - t0 * d
    t = t0 + step * torch.arange(N, dtype=torch.float32)[None].expand(p.shape[0], N)
    return o, d, t


def cam_to_world(c, pose):
    return c @ pose[:3, :3].T + pose[:3, 3]


def case_A():
    o, d = scattered_rays(77, 1)
    t, s = sample_t(o, d, 13, 2)
    return Case("A", (64, 48), 3, (24, 32), o, d, t, s, chunk=50, mlps=(0, 1, 2, 3))


def case_B():
    """256 scattered rays, then one 32-ray group (slots 256..287) whose 64 sample-0/1 points sit at the centres of 64 distinct
    boxes of the pitch-3 window lattice of view 0's xz plane: one job needs 64 texel windows of that map."""
    _, osc = scene((640, 480), 3, (120, 160))
    Hp, Wp = 120, 160
    o, d = scattered_rays(256, 3)
    t, s = sample_t(o, d, 4, 4)
    k = torch.arange(64)
    ix = 50 + 3 * (k % 8) + 1.5                          # texel-centre offsets: a one-texel fast-math shift cannot change the box
    iz = 5 + 3 * (k // 8) + 1.5
    g = torch.Generator().manual_seed(5)
    cam = torch.stack([2 * ix / (Wp - 1) - 1, (torch.rand(64, generator=g) - 0.5) * 0.2, 2 * iz / (Hp - 1) - 1], -1)
    p = cam_to_world(cam.double(), osc.src_poses[0].double()).float()
    a, b = p[0::2], p[1::2]                               # ray i: sample 0 at a_i, sample 1 at b_i
    dd = (b - a) / (b - a).norm(dim=-1, keepdim=True)
    oo = a - 0.05 * dd
    L = (b - a).norm(dim=-1)
    tt = torch.stack([torch.full_like(L, 0.05), 0.05 + L, 0.1 + L, 0.15 + L], -1)
    ss = torch.sort(torch.rand(32, 4, generator=g), -1, descending=True).values
    return Case("B", (640, 480), 3, (120, 160), torch.cat([o, oo]), torch.cat([d, dd]), torch.cat([t, tt]), torch.cat([s, ss]))


def case_C():
    fo, fd = frame_rays(6, 4)
    so, sd = scattered_rays(40, 6)
    o, d = torch.cat([fo, so]), torch.cat([fd, sd])
    t, s = sample_t(o, d, 6, 7)
    return Case("C", (6, 4), 2, (2, 2), o, d, t, s)


def case_D():
    fo, fd = frame_rays(37, 23)
    so, sd = scattered_rays(40, 8)
    o, d = torch.cat([fo[300:360], so]), torch.cat([fd[300:360], sd])
    t, s = sample_t(o, d, 9, 9)
    return Case("D", (37, 23), 5, (23, 37), o, d, t, s, chunk=64)


def case_E():
    o, d = scattered_rays(70, 10)
    t, s = sample_t(o, d, 5, 11)
    return Case("E", (64, 48), 8, (24, 32), o, d, t, s)


def case_F():
    """fg points of A's scene placed on texel lines and the -1 / W-1 borders of view 0's xz plane and latent, points in view 0's
    camera plane (z ~ 0) and behind it."""
    s_, osc = scene((64, 48), 3, (24, 32))
    pose = osc.src_poses[0].double()
    Hp, Wp = 24, 32
    Hl, Wl = 24, 32
    edge = lambda n: torch.tensor([-1.0, -0.5, -1e-3, 0.0, 0.5, 1.0, 2.0, n - 2.0, n - 1.5, n - 1.0, n - 0.5, n - 1e-3], dtype=torch.float64)
    g = torch.Generator().manual_seed(12)
    pts = []
    # xz plane: (ix, iz) on the lines / borders, cam y small
    ix, iz = torch.meshgrid(edge(Wp), torch.tensor([0.0, 3.0, 4.5, 7.0, 7.5, 9.0], dtype=torch.float64), indexing="ij")
    cx, cz = 2 * ix.reshape(-1) / (Wp - 1) - 1, 2 * iz.reshape(-1) / (Hp - 1) - 1
    pts.append(torch.stack([cx, (torch.rand(cx.shape[0], generator=g, dtype=torch.float64) - 0.5) * 0.2, cz], -1))
    # latent: pixel coordinates on its lines / borders at depth z = -0.8
    ls = lambda n, img: n / (n - 1) * 2.0 / img
    ux, uy = torch.meshgrid(edge(Wl), edge(Hl)[::3], indexing="ij")
    gx, gy = 2 * ux.reshape(-1) / (Wl - 1) - 1, 2 * uy.reshape(-1) / (Hl - 1) - 1
    u, v = (gx + 1) / ls(Wl, 64), (gy + 1) / ls(Hl, 48)
    z = torch.full_like(u, -0.8)
    f = float(osc.focal)
    pts.append(torch.stack([-(u - osc.cx) / f * (z + 1e-9), (v - osc.cy) / f * (z + 1e-9), z], -1))
    # camera plane and behind the camera
    k = 12
    pts.append(torch.stack([(torch.rand(k, generator=g, dtype=torch.float64) - 0.5) * 0.6,
                            (torch.rand(k, generator=g, dtype=torch.float64) - 0.5) * 0.2, torch.full((k,), 1e-7, dtype=torch.float64)], -1))
    pts.append(torch.stack([(torch.rand(k, generator=g, dtype=torch.float64) - 0.5) * 0.4,
                            (torch.rand(k, generator=g, dtype=torch.float64) - 0.5) * 0.2, torch.full((k,), 0.1, dtype=torch.float64)], -1))
    p = cam_to_world(torch.cat(pts), pose).float()
    p = p[p.norm(dim=-1) < 0.97]
    o, d, t = rays_through(p, N=4)
    return Case("F", (64, 48), 3, (24, 32), o, d, t, torch.linspace(0.9, 0.1, 4).expand(p.shape[0], 4).contiguous(), mlps=(0, 2))


def case_G():
    a = case_A()
    a.name = "G"
    a.order = torch.randperm(77, generator=torch.Generator().manual_seed(13)).int()
    a.mlps = (0, 1)
    return a


CASES = {"A": case_A, "B": case_B, "C": case_C, "D": case_D, "E": case_E, "F": case_F, "G": case_G}


def model_for(case, mi, device=None, cls=tm.TCFieldModel):
    _, osc = scene(case.img_wh, case.nv, case.plane_hw, case.seed)
    return cls(osc, synth.make_mlp_params(case.seed), mi, device=device)


def model_out(case, mi, device=None, cls=tm.TCFieldModel):
    m = model_for(case, mi, device, cls)
    rgb, sig = m.field(case.o, case.d, case.d, case.far, case.t(mi), case.chunk, case.order)
    return rgb.cpu(), sig.cpu()


def gap(rgb, sig, rgb_ref, sig_ref):
    """(max |d rgb|, max |d sigma| / (1 + sigma)) in float64."""
    rgb, sig, rgb_ref, sig_ref = (x.detach().cpu().double() for x in (rgb, sig, rgb_ref, sig_ref))
    return float((rgb - rgb_ref).abs().max()), float(((sig - sig_ref).abs() / (1 + sig_ref.abs())).max())


# ---------------- CPU: the model ----------------

@pytest.mark.parametrize("nv", [1, 3, 8])
@pytest.mark.parametrize("mi", [0, 1])
def test_model_is_a_reassociation_of_the_oracle(nv, mi):
    """With fp16 rounding switched off the model equals neo360_oracle.field (fp64) over chunked Q1 to 1e-9: the projected maps, the
    folded head and the view-sum are exact re-associations of the reference."""
    _, osc = scene((32, 24), nv, (12, 16), 1)
    P = synth.make_mlp_params(2)
    o, d = scattered_rays(45, 3)
    t, s = sample_t(o, d, 7, 4)
    t = s if mi & 1 else t
    far = orc.intersect_sphere(o, d)[:, 0]
    f = lambda x: x.double()
    ref = tm.oracle_field(tm.scene64(osc), {k: f(v) for k, v in P.items()}, mi, f(o), f(d), f(d), f(far), f(t), chunk=20)
    got = tm.TCFieldModel(osc, P, mi, rnd=False).field(o, d, d, far, t, chunk=20)
    assert float((got[0] - ref[0]).abs().max()) <= 1e-9 and float((got[1] - ref[1]).abs().max()) <= 1e-9
    # ... and chunking matters (quirk Q1), so the comparison above does test the chunk handling
    one = tm.TCFieldModel(osc, P, mi, rnd=False).field(o, d, d, far, t, chunk=0)
    assert float((one[0] - got[0]).abs().max()) > 1e-4


def test_window_grouping_helper():
    """window_groups numbers the windows of a job by first appearance in row order (row = sample_in_pair * 32 + ray)."""
    B, N = 33, 2                     # 2 ray groups (the second holds one ray) x 2 half-jobs
    x0 = torch.full((1, B, N), 5, dtype=torch.long)
    y0 = torch.zeros((1, B, N), dtype=torch.long)
    x0[0, 3, 0], x0[0, 7, 0], x0[0, 0, 1] = 9, 8, 12          # box 1 (first seen at row 3), box 1 again, box 2 (row 32)
    w = torch.ones(1, B, N, 4)
    w[0, 1, 1] = 0                                            # dead row
    gr = tm.window_groups(x0, y0, w)
    assert gr["nwin"].tolist() == [[3, 0, 1, 0]]                # jobs (group, half): samples 2, 3 are padding
    assert gr["win"][0, 3, 0] == 1 and gr["win"][0, 7, 0] == 1 and gr["win"][0, 0, 1] == 2 and gr["win"][0, 1, 1] == -1
    assert gr["bx"][0, 3, 0] == 1 and gr["bx"][0, 7, 0] == 0 and gr["bx"][0, 0, 1] == 1
    order = torch.arange(B).flip(0).int()                     # ray 32 now shares the first job with rays 31..1
    gr = tm.window_groups(x0, y0, w, order)
    assert gr["job"][0, 32, 0] == 0 and gr["job"][0, 0, 0] == 2


# ---- mutations: plausible kernel bugs, injected into one stage of the model ----

class ClampBorder(tm.TCFieldModel):
    """a border tap reads the clamped edge texel instead of zero (a wrong out-of-bounds fill)."""
    def taps(self, gx, gy, H, W):
        ix, iy = ((gx + 1) / 2) * (W - 1), ((gy + 1) / 2) * (H - 1)
        x0, y0 = torch.floor(ix), torch.floor(iy)
        inr = (ix >= -1) & (ix < W) & (iy >= -1) & (iy < H)
        w = torch.stack([(x0 + 1 - ix) * (y0 + 1 - iy), (ix - x0) * (y0 + 1 - iy), (x0 + 1 - ix) * (iy - y0), (ix - x0) * (iy - y0)], -1)
        return x0.long(), y0.long(), tm.r16(w * inr[..., None], self.rnd)

    def blend(self, m, x0, y0, w, groups=None):
        pm = self.pmaps[m]
        _, H, W, _ = pm.shape
        v = torch.arange(self.nv).reshape(-1, 1, 1)
        return sum(pm[v, (y0 + dy).clamp(0, H - 1), (x0 + dx).clamp(0, W - 1)] * w[..., k, None]
                   for k, (dx, dy) in enumerate(((0, 0), (1, 0), (0, 1), (1, 1))))


class BoxOffByOne(tm.TCFieldModel):
    """xz-plane rows at box offset 2 are keyed to the next lattice box: their taps read texels 3 to the right."""
    needs_groups = True

    def blend(self, m, x0, y0, w, groups=None):
        if m == 1:
            x0 = torch.where(groups["bx"] == 2, x0 + 3, x0)
        return super().blend(m, x0, y0, w, groups)


class SwapNeSw(tm.TCFieldModel):
    """the ne and sw tap weights swapped."""
    def taps(self, gx, gy, H, W):
        x0, y0, w = super().taps(gx, gy, H, W)
        return x0, y0, w[..., [0, 2, 1, 3]]


class DropP3(tm.TCFieldModel):
    """the layer-3 (P3) half of the xy plane's lookups is lost."""
    def blend(self, m, x0, y0, w, groups=None):
        out = super().blend(m, x0, y0, w, groups)
        return torch.cat([out[..., :128], torch.zeros_like(out[..., 128:])], -1) if m == 2 else out


class DropB2(tm.TCFieldModel):
    """b2 (bias MMA of layer 2) is dropped."""
    def weights(self, p):
        W = super().weights(p)
        W["b2"] = torch.zeros_like(W["b2"])
        return W


class Q1Shift(tm.TCFieldModel):
    """the quirk-Q1 conditioning ray is (j - 1) mod B instead of j mod B."""
    def q1_dirs(self, dirs_cam, B, N, chunk):
        ch = chunk if chunk > 0 else B
        rolled = torch.cat([torch.roll(dirs_cam[:, c0:c0 + ch], 1, dims=1) for c0 in range(0, B, ch)], 1)
        return super().q1_dirs(rolled, B, N, chunk)


class MissingView(tm.TCFieldModel):
    """the last source view is left out of sum_v h3_v."""
    def head(self, h3, dmean):
        return super().head(h3[:-1], dmean)


class LostBatch(tm.TCFieldModel):
    """rows of the xz plane whose window index is >= kRing / 2 = 4 get no lookup (a lost second batch of windows)."""
    needs_groups = True

    def blend(self, m, x0, y0, w, groups=None):
        out = super().blend(m, x0, y0, w, groups)
        return out * (groups["win"] < 4)[..., None] if m == 1 else out


MUTATIONS = [ClampBorder, BoxOffByOne, SwapNeSw, DropP3, DropB2, Q1Shift, MissingView, LostBatch]


def case_suite():
    """The inputs of test_field_eval_tc_vs_oracle (level 0): 75 contiguous frame rays of the 64x48 scene, stratified samples."""
    fo, fd = frame_rays(64, 48)
    o, d = fo[1000:1075].contiguous(), fd[1000:1075].contiguous()
    far = orc.intersect_sphere(o, d)
    t, _ = orc.sample_fg(o, d, 16, torch.full_like(far, 1e-4), far)
    s, _, _ = orc.sample_bg(o, d, 16, far)
    return Case("suite", (64, 48), 3, (24, 32), o, d, t, s, mlps=(0, 1, 2, 3))


def test_mutations_exceed_the_tc_bound():
    """Each injected bug moves rgb or sigma by >= 3x the TC bound in at least one stress scenario (A, F: A's scene), so the
    kernel-vs-model test would catch it.  The report also gives each bug's effect on the inputs of test_field_eval_tc_vs_oracle
    and whether that test's bounds (rgb 2e-2, sigma 2e-2 + 2 %) would have let it through."""
    cases = [case_A(), case_F(), case_suite()]
    base = {(c.name, mi): model_out(c, mi) for c in cases for mi in c.mlps}
    print(f"\n{'mutation':<13}{'stress: rgb':>12}{'sigma':>10}{'x TC bound':>11}{'suite inputs: rgb':>19}{'sigma':>10}   passes 2e-2 there")
    for cls in MUTATIONS:
        worst = {}
        for c in cases:
            for mi in c.mlps:
                (r, s), (mr, ms) = model_out(c, mi, cls=cls), base[(c.name, mi)]
                key = "suite" if c.name == "suite" else "stress"
                rs = (float((r - mr).abs().max()), float(((s - ms).abs() - 0.02 * ms.abs()).max()) if key == "suite" else gap(r, s, mr, ms)[1])
                w = worst.get(key, (0.0, 0.0))
                worst[key] = (max(w[0], rs[0]), max(w[1], rs[1]))
        x = max(worst["stress"][0] / TC_RGB_BOUND, worst["stress"][1] / TC_SIGMA_BOUND)
        hidden = worst["suite"][0] < 2e-2 and worst["suite"][1] < 2e-2
        print(f"{cls.__name__:<13}{worst['stress'][0]:>12.2e}{worst['stress'][1]:>10.2e}{x:>11.0f}{worst['suite'][0]:>19.2e}"
              f"{worst['suite'][1]:>10.2e}   {'yes' if hidden else 'no'}")
        assert x >= 3.0, (cls.__name__, worst)


# ---------------- GPU: the kernel ----------------

@pytest.fixture(scope="module")
def cuda():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from neo360_b200 import build
    build.build()
    return torch.device("cuda:0")


def make_net(case, dev):
    from neo360_b200 import NeRF_TP
    s, _ = scene(case.img_wh, case.nv, case.plane_hw, case.seed)
    net = NeRF_TP(num_coarse_samples=8, num_fine_samples=4, num_src_views=case.nv).eval()
    net.load_state_dict(synth.make_mlp_params(case.seed))
    net = net.to(dev)
    net.set_scene(*[s[k].to(dev) for k in ("planes_xz", "planes_xy", "planes_yz", "latent", "src_poses", "src_focal", "src_c")],
                  s["img_wh"], precisions=["fp32", "tc"])
    return net


def field_eval(net, case, mi, precision, dev):
    """neo_field_eval through the C ABI (chunk and ray order set), into NaN-filled outputs with a 4 KB tail."""
    from neo360_b200 import _lib as L
    n, N = case.t(mi).shape
    o, d, far, t = (x.contiguous().to(dev) for x in (case.o, case.d, case.far, case.t(mi)))
    order = None if case.order is None else case.order.to(dev).contiguous()
    r = L.NeoRays()
    r.n_rays, r.chunk = n, case.chunk
    r.rays_o, r.rays_d, r.viewdirs = L.ptr(o), L.ptr(d), L.ptr(d)
    r.ray_order = None if order is None else order.data_ptr()
    rgb = torch.full((n * N * 3 + TAIL,), float("nan"), device=dev)
    sig = torch.full((n * N + TAIL,), float("nan"), device=dev)
    L.check(L.load().neo_field_eval(net._scene.handle, C.byref(r), L.ptr(far), L.ptr(t), N, mi, precision, L.ptr(rgb), L.ptr(sig),
                                    torch.cuda.current_stream().cuda_stream))
    net.check()
    rgb, sig = rgb.cpu(), sig.cpu()
    assert bool(torch.isfinite(rgb[:n * N * 3]).all()) and bool(torch.isfinite(sig[:n * N]).all()), "an output was not written"
    assert bool(torch.isnan(rgb[n * N * 3:]).all()) and bool(torch.isnan(sig[n * N:]).all()), "written past n * N"
    return rgb[:n * N * 3].reshape(n, N, 3), sig[:n * N].reshape(n, N, 1)


def coverage(case, mi, dev):
    """Max windows per job per map (latent, xz, xy, yz) and row counts that the scenario claims to reach."""
    m = model_for(case, mi, dev)
    f = lambda x: x.to(dev, torch.float64)
    g = tm.geometry(m.sc, bool(mi & 1), f(case.o), f(case.d), f(case.d), f(case.far), f(case.t(mi)))
    out = {"nwin": [], "base-1": 0, "edge": 0, "dead": 0}
    for gx, gy, H, W in g.grids:
        x0, y0, w = m.taps(gx, gy, H, W)
        gr = tm.window_groups(x0, y0, w, case.order)
        out["nwin"].append(int(gr["nwin"].max()))
        live = gr["win"] >= 0
        out["base-1"] += int((live & ((x0 == -1) | (y0 == -1))).sum())
        out["edge"] += int((live & ((x0 == W - 1) | (y0 == H - 1))).sum())
        out["dead"] += int((~live).sum())
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_tc_field_vs_model(cuda, name):
    """Per scenario and MLP: TC kernel vs the model (tight bound), fp32 CUDA path vs the fp64 oracle (5e-5), every output written and
    nothing past n * N, and the scenario reaches the paths it is meant for."""
    case = CASES[name]()
    net = make_net(case, cuda)
    _, osc = scene(case.img_wh, case.nv, case.plane_hw, case.seed)
    f = lambda x: x.to(cuda, torch.float64)
    P64 = {k: f(v) for k, v in synth.make_mlp_params(case.seed).items()}
    fails = []
    for mi in case.mlps:
        rgb, sig = field_eval(net, case, mi, 1, cuda)
        mr, ms = model_out(case, mi, cuda)
        g_tc = gap(rgb, sig, mr, ms)
        if case.nv <= 4:
            r32, s32 = field_eval(net, case, mi, 0, cuda)
            ref = tm.oracle_field(tm.scene64(osc, cuda), P64, mi, f(case.o), f(case.d), f(case.d), f(case.far), f(case.t(mi)), case.chunk)
            g32 = gap(r32, s32, *ref)
        else:                                        # the fp32 path is built for 1..4 views and says so
            with pytest.raises(RuntimeError, match="1..4 source views"):
                field_eval(net, case, mi, 0, cuda)
            g32 = (float("nan"), float("nan"))
        cov = coverage(case, mi, cuda)
        print(f"\n[{name} mlp {mi}] rays {case.o.shape[0]} N {case.t(mi).shape[1]} nv {case.nv}: TC vs model rgb {g_tc[0]:.2e} "
              f"(bound {TC_RGB_BOUND:.0e}) sigma {g_tc[1]:.2e} (bound {TC_SIGMA_BOUND:.0e}); fp32 vs oracle rgb {g32[0]:.2e} "
              f"sigma {g32[1]:.2e}; max windows/job/map {cov['nwin']}; live rows at base -1 {cov['base-1']}, at W-1 {cov['edge']}, "
              f"dead {cov['dead']}")
        if not (g_tc[0] <= TC_RGB_BOUND and g_tc[1] <= TC_SIGMA_BOUND):
            fails.append(("tc", mi, g_tc))
        b32 = FP32_BOUND * (2 if name == "B" else 1)
        if case.nv <= 4 and not (g32[0] <= b32 and g32[1] <= b32):
            fails.append(("fp32", mi, g32))
        # coverage claims (margins: fast-math geometry can move a boundary point by one texel)
        if name in ("A", "G"):
            assert max(cov["nwin"]) > 4 * 2 and case.o.shape[0] % 32 and case.t(mi).shape[1] % 4 and case.o.shape[0] % case.chunk
        if name == "B" and mi == 0:
            assert cov["nwin"][1] >= 60, cov
        if name == "F":
            assert cov["base-1"] > 10 and cov["edge"] > 10 and cov["dead"] > 10, cov
    if name == "C":
        assert case.plane_hw == (2, 2) and (case.img_wh[1] // 2) * (case.img_wh[0] // 2) == 6      # projection GEMM M = 4 and 6
    if name == "G":
        assert not torch.equal(case.order.long(), torch.arange(case.o.shape[0]))
    assert not fails, fails
