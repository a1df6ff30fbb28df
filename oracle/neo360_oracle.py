"""TEST INFRASTRUCTURE ONLY -- CPU restatement (oracle) of the NeO-360 ray-marching hot path.

This file is the checker for the CUDA path in `neo360_b200/`; it is never the thing shipped or
measured as the product.  Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s CPU-baseline /
`--impl reference` legs import it.  Nothing under `neo360_b200/` does.

PARITY PIN: every function below is checked against the UNMODIFIED reference (imported through
`oracle/ref_shim.py`) by `oracle/make_golden.py`, which also writes the golden vectors under
`tests/golden/`; `tests/test_oracle_golden.py` re-checks the oracle against those vectors wherever the
reference tree is absent (the GPU box).  The reference ships no tests / golden vectors of its own
(SURVEY.md section 4), so reference-generated fixtures are the pin.

All arithmetic is fp32 torch on CPU, written stage by stage in the order of SURVEY.md Appendix A.
Reference citations are `path:line` relative to the reference root.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor

# --------------------------------------------------------------------------------------------
# a1/a2  ray generation                                  datasets/ray_utils.py:84-104, 133-176
# --------------------------------------------------------------------------------------------


def ray_directions(H: int, W: int, focal: float) -> Tensor:
    """Camera-frame directions ((i-W/2)/f, -(j-H/2)/f, -1), no half-pixel offset (ray_utils.py:97-102)."""
    j, i = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32),
                          indexing="ij")
    return torch.stack([(i - W / 2) / focal, -(j - H / 2) / focal, -torch.ones_like(i)], -1)


def rays_from_pose(directions: Tensor, c2w: Tensor):
    """get_rays(..., output_view_dirs=True, output_radii=True) (ray_utils.py:133-171).

    Returns rays_o, viewdirs, rays_d, radii.  Quirk Q3: viewdirs aliases rays_d and is normalised in
    place (ray_utils.py:163-164), so rays_d comes back unit-norm as well."""
    d_raw = directions @ c2w[:, :3].T  # (H, W, 3)
    o = c2w[:, 3].expand(d_raw.shape)
    dx = torch.sqrt(torch.sum((d_raw[:-1] - d_raw[1:]) ** 2, dim=-1))
    dx = torch.cat([dx, dx[-2:-1]], dim=0)
    radii = (dx[..., None] * 2 / torch.sqrt(torch.tensor(12, dtype=torch.int8))).reshape(-1)
    d = d_raw / torch.norm(d_raw, dim=-1, keepdim=True)
    d = d.reshape(-1, 3)
    return o.reshape(-1, 3).contiguous(), d, d, radii


def sample_training_rays(pix_inds: Tensor, H: int, W: int, focal: float, poses: Tensor, images: Tensor = None):
    """The pixel sampling of the training `__getitem__` (datasets/nerds360_ae.py:684-748): every ray of every target view is built,
    stacked (T, H*W, .), flattened and indexed by `pix_inds`.  Returns rays_o, viewdirs, rays_d, radii (n,1), target (n,3) or None."""
    dirs = ray_directions(H, W, focal)
    per_view = [rays_from_pose(dirs, c2w[:3, :4]) for c2w in poses]
    o, vd, rd, radii = (torch.stack([v[k] for v in per_view], 0) for k in range(4))
    tgt = None if images is None else images.reshape(-1, 3)[pix_inds]
    return o.reshape(-1, 3)[pix_inds], vd.reshape(-1, 3)[pix_inds], rd.reshape(-1, 3)[pix_inds], radii.reshape(-1, 1)[pix_inds], tgt


# --------------------------------------------------------------------------------------------
# a3  ray / unit-sphere intersection                         models/neo360/helper.py:253-273
# --------------------------------------------------------------------------------------------


def intersect_sphere(o: Tensor, d: Tensor) -> Tensor:
    d1 = -(d * o).sum(-1, keepdim=True) / (d * d).sum(-1, keepdim=True)
    p = o + d1 * d
    inv_norm = 1.0 / torch.norm(d, dim=-1, keepdim=True)
    p2 = (p * p).sum(-1, keepdim=True)
    if not bool(torch.all(1.0 - p2 >= 0)):  # helper.py:271 (assert)
        raise AssertionError("1.0 - p_norm_sq should be greater than 0")
    return d1 + torch.sqrt(1.0 - p2) * inv_norm


# --------------------------------------------------------------------------------------------
# a5  inverted-sphere parametrisation                       models/neo360/helper.py:401-450
# --------------------------------------------------------------------------------------------


def depth2pts_outside(o: Tensor, d: Tensor, s: Tensor) -> Tensor:
    """o,d (B,3); s (B,N) inverse radius in [0,1]  ->  (B,N,4) = (unit point, s)."""
    o = o[:, None, :].expand(*s.shape, 3)
    d = d[:, None, :].expand(*s.shape, 3)
    d1 = -(d * o).sum(-1, keepdim=True) / (d * d).sum(-1, keepdim=True)
    p_mid = o + d1 * d
    rho = torch.norm(p_mid, dim=-1, keepdim=True)
    inv_norm = 1.0 / torch.norm(d, dim=-1, keepdim=True)
    if not bool(torch.all(1.0 - rho * rho >= 0)):  # helper.py:426
        raise AssertionError("1.0 - p_mid_norm * p_mid_norm should be greater than 0")
    d2 = torch.sqrt(1.0 - rho * rho) * inv_norm
    p_sph = o + (d1 + d2) * d
    axis = torch.cross(o, p_sph, dim=-1)
    axis = axis / torch.norm(axis, dim=-1, keepdim=True)
    phi = torch.asin(rho)
    theta = torch.asin(rho * s[..., None])
    ang = phi - theta
    p_new = (p_sph * torch.cos(ang) + torch.cross(axis, p_sph, dim=-1) * torch.sin(ang)
             + axis * (axis * p_sph).sum(-1, keepdim=True) * (1.0 - torch.cos(ang)))
    p_new = p_new / (torch.norm(p_new, dim=-1, keepdim=True) + 1e-10)
    return torch.cat([p_new, s[..., None]], dim=-1)


# --------------------------------------------------------------------------------------------
# a4  stratified sampling                                     models/neo360/helper.py:24-75
# --------------------------------------------------------------------------------------------


def _jitter(t: Tensor, u_rand: Tensor) -> Tensor:
    mids = 0.5 * (t[..., 1:] + t[..., :-1])
    upper = torch.cat([mids, t[..., -1:]], -1)
    lower = torch.cat([t[..., :1], mids], -1)
    return lower + (upper - lower) * u_rand


def sample_fg(o, d, n, near, far, u_rand: Optional[Tensor] = None):
    """in_sphere=True branch.  u_rand (B,n+1) replaces torch.rand (helper.py:50) when randomized."""
    u = torch.linspace(0.0, 1.0, n + 1, device=o.device)
    t = near * (1.0 - u) + far * u
    if u_rand is not None:
        t = _jitter(t, u_rand)
    else:
        t = torch.broadcast_to(t, (o.shape[0], n + 1))
    pts = o[:, None, :] + t[..., None] * d[:, None, :]
    return t, pts


def sample_bg(o, d, n, far, far_unc=3.0, u_rand: Optional[Tensor] = None):
    """in_sphere=False branch: s descends 1->0; `lin` are the farthest-first lookup points (quirk Q2)."""
    B = o.shape[0]
    s = torch.broadcast_to(torch.linspace(0.0, 1.0, n + 1, device=o.device), (B, n + 1))
    if u_rand is not None:
        s = _jitter(s, u_rand)
    t_lin = far * (1.0 - s) + far_unc * s
    s = torch.flip(s, dims=[-1])
    t_lin = torch.flip(t_lin, dims=[-1])
    lin = o[:, None, :] + t_lin[..., None] * d[:, None, :]
    return s, depth2pts_outside(o, d, s), lin


# --------------------------------------------------------------------------------------------
# a14/a15  inverse-CDF resampling                          models/neo360/helper.py:174-249
# --------------------------------------------------------------------------------------------


def piecewise_constant_pdf(bins: Tensor, w: Tensor, m: int, u_rand: Optional[Tensor] = None) -> Tensor:
    """bins (B,K), w (B,K-1) -> (B,m).  Bracketing is by VALUE max/min under the compare mask
    (helper.py:204-210), which matters for the descending bg bins (quirk Q17)."""
    eps = 1e-5
    wsum = w.sum(-1, keepdim=True)
    pad = torch.fmax(torch.zeros_like(wsum), eps - wsum)
    w = w + pad / w.shape[-1]
    wsum = wsum + pad
    pdf = w / wsum
    cdf = torch.fmin(torch.ones_like(pdf[..., :-1]), torch.cumsum(pdf[..., :-1], -1))
    cdf = torch.cat([torch.zeros_like(cdf[..., :1]), cdf, torch.ones_like(cdf[..., :1])], -1)
    if u_rand is not None:
        u = u_rand
    else:
        u = torch.linspace(0.0, 1.0 - 2 ** -32, m, device=w.device)  # endpoint rounds to 1.0 in fp32 (quirk Q7)
        u = torch.broadcast_to(u, (*cdf.shape[:-1], m))
    mask = u[..., None, :] >= cdf[..., :, None]

    def lo(x):
        return (mask * x[..., None] + ~mask * x[..., :1, None]).max(-2)[0]

    def hi(x):
        return (~mask * x[..., None] + mask * x[..., -1:, None]).min(-2)[0]

    b0, b1, c0, c1 = lo(bins), hi(bins), lo(cdf), hi(cdf)
    tau = torch.clip(torch.nan_to_num((u - c0) / (c1 - c0), 0), 0, 1)
    return b0 + tau * (b1 - b0)


def fg_points(o, d, t):
    """fg sample points o + t d for t (B,N) (helper.py:52-53)."""
    return o[:, None, :] + t[..., None] * d[:, None, :]


def bg_points(o, d, s, far, far_unc=3.0):
    """bg points for inverse radii s (B,N): the unit-sphere points fed to the encoding and the lookup points
    o + (far (1-s) + far_unc s) d (quirk Q2)."""
    t_lin = far * (1.0 - s) + far_unc * s
    return depth2pts_outside(o, d, s), o[:, None, :] + t_lin[..., None] * d[:, None, :]


def resample_fg(o, d, t_old, w, m, u_rand=None):
    mids = 0.5 * (t_old[..., 1:] + t_old[..., :-1])
    t_new = piecewise_constant_pdf(mids, w[..., 1:-1], m, u_rand).detach()      # helper.py:222-224: no gradient through the new samples
    t = torch.sort(torch.cat([t_old, t_new], -1), -1).values
    return t, fg_points(o, d, t)


def resample_bg(o, d, s_old, w, m, far, far_unc=3.0, u_rand=None):
    mids = 0.5 * (s_old[..., 1:] + s_old[..., :-1])
    s_new = piecewise_constant_pdf(mids, w[..., 1:-1], m, u_rand).detach()      # helper.py:222-224
    s = torch.flip(torch.sort(torch.cat([s_old, s_new], -1), -1).values, dims=[-1])
    return (s, *bg_points(o, d, s, far, far_unc))


# --------------------------------------------------------------------------------------------
# a6  world -> source-camera frames                       models/neo360/util.py:45-70
# --------------------------------------------------------------------------------------------


def world2camera(x: Tensor, c2w: Tensor) -> Tensor:
    """x (M,3); c2w (NV,4,4)  ->  (NV,M,3) = R^T x + (-(R^T t)) in that order (util.py:64-68)."""
    rot = c2w[:, :3, :3].transpose(1, 2)
    trans = -torch.bmm(rot, c2w[:, :3, 3:])
    return torch.matmul(rot[:, None], x[None, :, :, None])[..., 0] + trans[:, None, :, 0]


def world2camera_dirs(v: Tensor, c2w: Tensor) -> Tensor:
    rot = c2w[:, :3, :3].transpose(1, 2)
    return torch.matmul(rot[:, None], v[None, :, :, None])[..., 0]


# --------------------------------------------------------------------------------------------
# a7/a8  bilinear lookups                encoder_tp_fusion_conv.py:122-209, encoder_pn.py:101-152
# --------------------------------------------------------------------------------------------


def bilinear_zeros(fmap: Tensor, gx: Tensor, gy: Tensor, impl: str = "explicit") -> Tensor:
    """F.grid_sample(fmap, [gx,gy], bilinear, align_corners=True, padding_mode='zeros') restated.
    fmap (NV,C,H,W); gx,gy (NV,M)  ->  (NV,M,C).  `impl='aten'` calls the same ATen op the reference
    calls (used for the timed CPU baseline); 'explicit' is the 4-tap gather restatement."""
    NV, C, H, W = fmap.shape
    if impl == "aten":
        g = torch.stack([gx, gy], -1)[:, :, None, :]
        return F.grid_sample(fmap, g, mode="bilinear", padding_mode="zeros", align_corners=True)[..., 0] \
            .permute(0, 2, 1)
    x0, y0, w = bilinear_quad(gx, gy, H, W)
    flat = fmap.reshape(NV, C, H * W).permute(0, 2, 1)  # (NV, HW, C)

    def tap(xx, yy, ww):
        idx = (yy.clamp(0, H - 1) * W + xx.clamp(0, W - 1)).long()
        val = torch.gather(flat, 1, idx[..., None].expand(-1, -1, C))
        return val * ww[..., None]

    return tap(x0, y0, w[..., 0]) + tap(x0 + 1, y0, w[..., 1]) + tap(x0, y0 + 1, w[..., 2]) + tap(x0 + 1, y0 + 1, w[..., 3])


def bilinear_quad(gx: Tensor, gy: Tensor, H: int, W: int):
    """The 2x2 tap quad of grid_sample(bilinear, align_corners=True, zeros): base texel (x0, y0) (floats, unclamped) and the
    weights (..., 4) of nw, ne, sw, se, zero for a tap outside the map."""
    ix = ((gx + 1) / 2) * (W - 1)
    iy = ((gy + 1) / 2) * (H - 1)
    x0 = torch.floor(ix)
    y0 = torch.floor(iy)
    x1 = x0 + 1
    y1 = y0 + 1
    ok = lambda xx, yy: (xx >= 0) & (xx <= W - 1) & (yy >= 0) & (yy <= H - 1)
    w = torch.stack([(x1 - ix) * (y1 - iy) * ok(x0, y0), (ix - x0) * (y1 - iy) * ok(x1, y0),
                     (x1 - ix) * (iy - y0) * ok(x0, y1), (ix - x0) * (iy - y0) * ok(x1, y1)], -1)
    return x0, y0, w


@dataclass
class Scene:
    """What the (out-of-scope) encoder hands to the hot path, plus the source cameras."""
    planes_xz: Tensor  # (NV,128,Hp,Wp)   encoder_tp_fusion_conv.py:585-595
    planes_xy: Tensor
    planes_yz: Tensor
    latent: Tensor     # (NV,512,Hl,Wl)   encoder_pn.py:203
    src_poses: Tensor  # (NV,4,4) camera-to-world
    focal: float       # src_focal[0]     model.py:242
    cx: float          # src_c[0]         model.py:244
    cy: float
    img_w: int         # src_imgs.shape[-1]   model.py:267-269
    img_h: int


def triplane_lookup(p_cam: Tensor, sc: Scene, impl="explicit") -> Tensor:
    """index_grid: sum of three plane lookups at camera-frame coords used directly as grid coords."""
    x, y, z = p_cam[..., 0], p_cam[..., 1], p_cam[..., 2]
    return (bilinear_zeros(sc.planes_xz, x, z, impl) + bilinear_zeros(sc.planes_xy, x, y, impl)
            + bilinear_zeros(sc.planes_yz, y, z, impl))


def local_lookup(p_cam: Tensor, sc: Scene, impl="explicit") -> Tensor:
    """get_local_feats (model.py:239-264) -> projection (util.py:92-111) -> index (encoder_pn.py:101-152)."""
    gx, gy = local_coords(p_cam, sc)
    return bilinear_zeros(sc.latent, gx, gy, impl)


def local_coords(p_cam: Tensor, sc: Scene):
    """Grid coordinates of the camera-frame points in the pixel-aligned latent (util.py:92-111, encoder_pn.py:116-120)."""
    uv = -p_cam[..., :2] / (p_cam[..., 2:] + 1e-9)
    dev = p_cam.device
    uv = uv * torch.tensor([sc.focal, -sc.focal], device=dev) + torch.tensor([sc.cx, sc.cy], device=dev)
    Hl, Wl = sc.latent.shape[-2:]
    ls = torch.tensor([float(Wl), float(Hl)], device=dev)
    ls = ls / (ls - 1) * 2.0
    scale = ls / torch.tensor([float(sc.img_w), float(sc.img_h)], device=dev)
    uv = uv * scale - 1.0
    return uv[..., 0], uv[..., 1]


# --------------------------------------------------------------------------------------------
# a9  positional encoding                                    models/neo360/helper.py:121-125
# --------------------------------------------------------------------------------------------


def pos_enc(x: Tensor, min_deg: int, max_deg: int) -> Tensor:
    scales = torch.tensor([2.0 ** i for i in range(min_deg, max_deg)], dtype=x.dtype, device=x.device)
    xb = (x[..., None, :] * scales[:, None]).reshape(*x.shape[:-1], -1)
    return torch.cat([x, torch.sin(torch.cat([xb, xb + 0.5 * math.pi], -1))], -1)


# --------------------------------------------------------------------------------------------
# a10/a11  conditioned MLP + activations               models/neo360/model.py:110-158, 343-407
# --------------------------------------------------------------------------------------------


def mlp_forward(P: Dict[str, Tensor], pre: str, enc: Tensor, dir_tile: Tensor, world: Tensor, local: Tensor,
                nv: int):
    """enc (NV,M,63|84); dir_tile (NV*M,27); world (NV*M,128); local (NV*M,512) -> raw rgb (M,3), raw sigma (M,1)."""
    M = enc.shape[1]
    lin = lambda name, x: F.linear(x, P[pre + name + ".weight"], P[pre + name + ".bias"])
    inp = torch.cat([enc.reshape(-1, enc.shape[-1]), local, world], -1)
    h = torch.relu(lin("pts_linears.0", inp))
    h = torch.relu(lin("pts_linears.1", h))
    h = torch.relu(lin("pts_linears.2", h))
    h = torch.relu(lin("pts_linears.3", torch.cat([h, inp], -1)))
    beta = lin("bottleneck_layer", h)
    hbar = h.reshape(nv, M, -1).mean(0)
    raw_sigma = lin("density_layer", hbar)
    q = lin("views_linear.0", torch.cat([beta, dir_tile], -1)).reshape(nv, M, -1).mean(0)
    q = torch.relu(lin("views_linear.1", torch.relu(q)))
    return lin("rgb_layer", q), raw_sigma


def field(P, pre, pts_cam_enc_in: Tensor, dirs_cam: Tensor, world, local, B: int, N: int, nv: int):
    """`predict` closure.  pts_cam_enc_in (NV,B*N,3|4); dirs_cam (NV,B,3).  Quirk Q1: the direction
    encoding is tiled along the RAY axis, so row j=b*N+s sees ray (j mod B)."""
    enc = pos_enc(pts_cam_enc_in, 0, 10)
    denc = pos_enc(dirs_cam, 0, 4)                       # (NV,B,27)
    dir_tile = q1_dir_tile(denc, N)
    raw_rgb, raw_sigma = mlp_forward(P, pre, enc, dir_tile, world, local, nv)
    sigma = F.softplus(raw_sigma.reshape(B, N, 1) - 1.0)
    rgb = torch.sigmoid(raw_rgb.reshape(B, N, 3)) * (1 + 2 * 0.001) - 0.001
    return rgb, sigma


def q1_dir_tile(denc: Tensor, N: int) -> Tensor:
    """(NV,B,C) -> (NV*B*N, C): the reference tiles the direction encoding along the RAY axis (model.py:357-360), so row
    j = b*N+s of each view is conditioned on ray (j mod B) of the batch (quirk Q1)."""
    return denc[:, None].repeat(1, 1, N, 1).reshape(-1, denc.shape[-1])


# --------------------------------------------------------------------------------------------
# a12  alpha compositing                                    models/neo360/helper.py:128-171
# --------------------------------------------------------------------------------------------


def composite(rgb, sigma, t, d, white_bkgd: bool, in_sphere: bool, t_far=None):
    if in_sphere:
        dist = torch.cat([t[..., 1:] - t[..., :-1], t_far - t[..., -1:]], -1)
        dist = dist * torch.norm(d[..., None, :], dim=-1)
    else:
        dist = torch.cat([t[..., :-1] - t[..., 1:], torch.full_like(t[..., :1], 1e10)], -1)
    alpha = 1.0 - torch.exp(-sigma[..., 0] * dist)
    T = torch.cumprod(1.0 - alpha + 1e-10, -1)           # quirk Q9: eps inside the product
    lam = T[..., -1:] if in_sphere else None
    w = alpha * torch.cat([torch.ones_like(T[..., -1:]), T[..., :-1]], -1)
    acc = w.sum(-1)
    out = (w[..., None] * rgb).sum(-2)
    if white_bkgd:
        out = out + (1.0 - acc[..., None])
    depth = (w * t).sum(-1)
    return out, acc, w, lam, depth


# --------------------------------------------------------------------------------------------
# a16  two-level fg/bg renderer                             models/neo360/model.py:266-581
# --------------------------------------------------------------------------------------------

MLP_NAMES = ("fg_coarse_mlp.", "bg_coarse_mlp.", "fg_fine_mlp.", "bg_fine_mlp.")


def render(rays: Dict[str, Tensor], sc: Scene, P: Dict[str, Tensor], n_coarse: int, n_fine: int,
           white_bkgd: bool = False, out_depth: bool = True, rand: Optional[Dict[str, Tensor]] = None,
           lookup_impl: str = "explicit", return_aux: bool = False):
    """NeRF_TP.forward with the encoder hoisted (its outputs are `sc`).  `rand`, if given, supplies the
    uniforms the reference would draw: keys fg0,bg0 (B,n_coarse+1) and fg1,bg1 (B,n_fine)."""
    o, d, vd = rays["rays_o"], rays["rays_d"], rays["viewdirs"]
    B = o.shape[0]
    nv = sc.src_poses.shape[0]
    near = torch.full_like(o[..., -1:], 1e-4)            # quirk Q4: near/far arguments ignored
    far = intersect_sphere(o, d)
    dirs_cam = world2camera_dirs(vd, sc.src_poses)
    ret, aux = [], []
    fg_w = bg_w = fg_t = bg_s = None
    for level in range(2):
        r = (lambda k: None if rand is None else rand.get(k))
        if level == 0:
            fg_t, fg_pts = sample_fg(o, d, n_coarse, near, far, r("fg0"))
            bg_s, bg_pts, bg_lin = sample_bg(o, d, n_coarse, far, 3.0, r("bg0"))
        else:
            fg_t, fg_pts = resample_fg(o, d, fg_t, fg_w, n_fine, r("fg1"))
            bg_s, bg_pts, bg_lin = resample_bg(o, d, bg_s, bg_w, n_fine, far, 3.0, r("bg1"))
        N = fg_t.shape[1]
        fg_pre, bg_pre = MLP_NAMES[2 * level], MLP_NAMES[2 * level + 1]
        fg_cam = world2camera(fg_pts.reshape(-1, 3), sc.src_poses)
        lin_cam = world2camera(bg_lin.reshape(-1, 3), sc.src_poses)
        bg_cam = world2camera(bg_pts[..., :3].reshape(-1, 3), sc.src_poses)
        bg_cam4 = torch.cat([bg_cam, bg_pts[..., 3].reshape(1, -1, 1).repeat(nv, 1, 1)], -1)
        fg_rgb, fg_sig = field(P, fg_pre, fg_cam, dirs_cam,
                               triplane_lookup(fg_cam, sc, lookup_impl).reshape(-1, 128),
                               local_lookup(fg_cam, sc, lookup_impl).reshape(-1, sc.latent.shape[1]), B, N, nv)
        bg_rgb, bg_sig = field(P, bg_pre, bg_cam4, dirs_cam,
                               triplane_lookup(lin_cam, sc, lookup_impl).reshape(-1, 128),
                               local_lookup(lin_cam, sc, lookup_impl).reshape(-1, sc.latent.shape[1]), B, N, nv)
        wb = False if out_depth else white_bkgd          # model.py:501,519 vs 551,560
        fg_c, fg_acc, fg_w, lam, fg_depth = composite(fg_rgb, fg_sig, fg_t, d, wb, True, far)
        bg_c, bg_acc, bg_w, _, bg_depth = composite(bg_rgb, bg_sig, bg_s, d, wb, False)
        comp = fg_c + lam * bg_c
        if out_depth:
            ret.append((comp, fg_c, bg_c, fg_acc, lam, fg_depth + lam.squeeze(-1) * bg_depth))
        else:
            fg_m = 0.5 * (fg_t[..., 1:] + fg_t[..., :-1])
            fg_m = torch.cat([fg_m, (fg_m[:, -1] + (fg_m[:, -1] - fg_m[:, -2]))[:, None]], -1)
            bg_m = torch.cat([0.5 * (bg_s[..., 1:] + bg_s[..., :-1]), bg_s[..., -1:]], -1)
            ret.append((comp, fg_w, bg_w, fg_m, bg_m, bg_acc))
        aux.append(dict(fg_t=fg_t, bg_s=bg_s, fg_rgb=fg_rgb, fg_sigma=fg_sig, bg_rgb=bg_rgb, bg_sigma=bg_sig,
                        fg_w=fg_w, bg_w=bg_w, far=far))
    return (ret, aux) if return_aux else ret


def render_chunked(rays, sc, P, n_coarse, n_fine, chunk=1024, **kw):
    """render_rays_test's chunk loop (model.py:861-896): keeps level-1 comp_rgb/fg/bg/depth."""
    B = rays["rays_o"].shape[0]
    keep = {"comp_rgb": [], "fg_rgb": [], "bg_rgb": [], "depth": [], "fg_acc": []}
    for i in range(0, B, chunk):
        sub = {k: v[i:i + chunk] for k, v in rays.items()}
        out = render(sub, sc, P, n_coarse, n_fine, white_bkgd=False, out_depth=True, **kw)[1]
        keep["comp_rgb"].append(out[0]); keep["fg_rgb"].append(out[1]); keep["bg_rgb"].append(out[2])
        keep["fg_acc"].append(out[3]); keep["depth"].append(out[5])
    return {k: torch.cat(v, 0) for k, v in keep.items()}


def psnr(pred: Tensor, gt: Tensor) -> float:
    """models/interface.py:53-61 (clip to [0,1], -10 log10 mse)."""
    mse = torch.mean((pred.clip(0, 1) - gt.clip(0, 1)) ** 2)
    return float(-10.0 * torch.log(mse) / math.log(10)) if mse > 0 else float("inf")
