"""TEST INFRASTRUCTURE ONLY -- a restatement of the ARITHMETIC of the tensor-core field kernel (neo360_b200/csrc/field_tc.cu).

`neo_field_eval(precision=NEO_PREC_TC)` evaluates the reference's radiance field re-associated (DESIGN.md section 5): the latent
columns of layers 0 and 3 are applied to the feature maps once per scene, the bilinear lookups blend those projected maps, and the
bottleneck / view-mean / views_linear.0 chain is folded into one head matrix.  Operands are fp16, accumulation is fp32.  This
module computes the same thing in fp64 and rounds to fp16 (round to nearest even, as `__float2half_rn`) at exactly the points
where the kernel rounds, so the kernel can be held to a bound set by fp32 accumulation order and fast-math geometry instead of
one that has to absorb fp16 operand rounding.  With `rnd=False` nothing is rounded and the model is an exact re-association of
`neo360_oracle.field`.

Rounding points (field_tc.cu):
  * projected maps  P = fp16(fp16(F) . fp16(Wsel)^T), Wsel = [W0 | W3] map columns (tc_scene_create, wsel_kernel, gemm_f16);
  * tap weights     fp16 of tap_quad's bilinear weights (geometry warps -> ROWINFO);
  * encoding        fp16 of the positional encoding with a constant-one column, so b0 / b3 enter as fp16 weights (enc_cols,
                    wimg_kernel); W0enc, W1, W2, W3h, W3enc fp16.  The kernel evaluates the sines with __sinf and a double-angle
                    recurrence whose error doubles per level; the model uses exact sin / cos, which is most of the gap below;
  * trunk           b1, b2 fp16 through the bias MMA; after every layer h = relu(fp16(pre-activation)) (epilogue);
  * head            Whead_h = fp16(fp32(Wv0[:, :128] . Wb) / nv), wsig / nv fp16, applied to sum_v h3_v in fp32 and never rounded;
                    direction term fp16(Wv0[:, 128:]) . fp16(mean_v enc(dir_v)) of the quirk-Q1 ray of the caller's chunk; + bq
                    (fp32), relu, fp16; views_linear.1 (fp16 weights, fp32 bias), relu, fp16; rgb_layer; sigmoid * 1.002 - 0.001;
                    sigma = softplus(raw - 1) with threshold 20 (head_kernel, head_stage).

The stages are methods of `TCFieldModel` so a test can replace one of them (tests/test_tc_field_stress.py injects kernel bugs
that way).  `window_groups` applies the kernel's texel-window grouping rule to the same geometry.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional

import torch
import torch.nn.functional as F

from oracle import neo360_oracle as orc

Tensor = torch.Tensor
MAPS = ("latent", "xz", "xy", "yz")
TILE_RAYS, TILE_SAMPLES, HALF_PTS, PITCH = 32, 4, 64, 3      # field_tc.cu: kTileRays, kTileSamples, kHalfPts; window lattice pitch


def r16(x: Tensor, on: bool = True) -> Tensor:
    """Round to fp16 (nearest even) and back to x's dtype."""
    return x.half().to(x.dtype) if on else x


def scene64(sc: orc.Scene, device=None) -> orc.Scene:
    """The oracle scene in fp64 (on `device`)."""
    t = lambda x: x.to(device=device, dtype=torch.float64)
    return orc.Scene(t(sc.planes_xz), t(sc.planes_xy), t(sc.planes_yz), t(sc.latent), t(sc.src_poses), sc.focal, sc.cx, sc.cy,
                     sc.img_w, sc.img_h)


@dataclass
class Geometry:
    enc_in: Tensor          # (nv, B, N, 3|4) camera-frame point fed to the positional encoding (+ s for bg)
    look_cam: Tensor        # (nv, B*N, 3) camera-frame lookup point (fg: the sample point, bg: the quirk-Q2 point)
    grids: List[tuple]      # per map (latent, xz, xy, yz): (gx, gy, H, W), gx / gy (nv, B, N)
    dirs_cam: Tensor        # (nv, B, 3) view directions in the source cameras


def geometry(sc: orc.Scene, is_bg: bool, o: Tensor, d: Tensor, vd: Tensor, far: Tensor, t: Tensor) -> Geometry:
    """Sample points, their source-camera coordinates and the grid coordinates of the four maps, all through the oracle."""
    nv = sc.src_poses.shape[0]
    B, N = t.shape
    if is_bg:
        xhat, lin = orc.bg_points(o, d, t, far.reshape(B, 1))
        enc_pt, look = xhat[..., :3], lin
    else:
        enc_pt = look = orc.fg_points(o, d, t)
    cam = orc.world2camera(enc_pt.reshape(-1, 3), sc.src_poses)
    enc_in = torch.cat([cam, t.reshape(1, -1, 1).expand(nv, -1, 1)], -1) if is_bg else cam
    lc = orc.world2camera(look.reshape(-1, 3), sc.src_poses) if is_bg else cam
    shp = lambda a: a.reshape(nv, B, N)
    gl = orc.local_coords(lc, sc)
    Hl, Wl = sc.latent.shape[-2:]
    Hp, Wp = sc.planes_xz.shape[-2:]
    x, y, z = lc[..., 0], lc[..., 1], lc[..., 2]
    grids = [(shp(gl[0]), shp(gl[1]), Hl, Wl), (shp(x), shp(z), Hp, Wp), (shp(x), shp(y), Hp, Wp), (shp(y), shp(z), Hp, Wp)]
    return Geometry(enc_in.reshape(nv, B, N, -1), lc, grids, orc.world2camera_dirs(vd, sc.src_poses))


def oracle_field(sc: orc.Scene, P: Dict[str, Tensor], mlp_index: int, o, d, vd, far, t, chunk: int = 0):
    """`neo360_oracle.field` over the caller's chunks (quirk Q1 ties each ray to its chunk): what neo_field_eval computes in the
    reference formulation.  Returns rgb (B, N, 3), sigma (B, N, 1) in the dtype of the inputs."""
    pre = orc.MLP_NAMES[mlp_index]
    nv = sc.src_poses.shape[0]
    B, N = t.shape
    ch = chunk if chunk > 0 else B
    rgb, sig = [], []
    for c0 in range(0, B, ch):
        s = slice(c0, min(c0 + ch, B))
        g = geometry(sc, bool(mlp_index & 1), o[s], d[s], vd[s], far[s], t[s])
        Bc = t[s].shape[0]
        world = orc.triplane_lookup(g.look_cam, sc).reshape(-1, 128)
        local = orc.local_lookup(g.look_cam, sc).reshape(-1, sc.latent.shape[1])
        a, b = orc.field(P, pre, g.enc_in.reshape(nv, Bc * N, -1), g.dirs_cam, world, local, Bc, N, nv)
        rgb.append(a); sig.append(b)
    return torch.cat(rgb), torch.cat(sig)


class TCFieldModel:
    """What `neo_field_eval(precision=NEO_PREC_TC)` computes for one MLP, in fp64 with the kernel's fp16 rounding points."""

    def __init__(self, sc: orc.Scene, P: Dict[str, Tensor], mlp_index: int, rnd: bool = True, device=None):
        self.sc = scene64(sc, device)
        self.dev = self.sc.latent.device
        self.rnd = rnd
        self.mlp_index = mlp_index
        self.is_bg = bool(mlp_index & 1)
        self.nv = self.sc.src_poses.shape[0]
        pre = orc.MLP_NAMES[mlp_index]
        p = {k[len(pre):]: v.to(self.dev, torch.float64) for k, v in P.items() if k.startswith(pre)}
        self.W = self.weights(p)
        self.pmaps = self.project(p)

    # ---- per-scene preparation ----
    def weights(self, p):
        q = lambda x: r16(x, self.rnd)
        E = 84 if self.is_bg else 63
        w0, w3, wv0 = p["pts_linears.0.weight"], p["pts_linears.3.weight"], p["views_linear.0.weight"]
        nv = self.nv
        return dict(
            W0enc=q(w0[:, :E]), b0=q(p["pts_linears.0.bias"]), W1=q(p["pts_linears.1.weight"]), b1=q(p["pts_linears.1.bias"]),
            W2=q(p["pts_linears.2.weight"]), b2=q(p["pts_linears.2.bias"]), W3h=q(w3[:, :128]), W3enc=q(w3[:, 128:128 + E]),
            b3=q(p["pts_linears.3.bias"]),
            Whh=q((wv0[:, :128] @ p["bottleneck_layer.weight"]) / nv), wsig=q(p["density_layer.weight"][0] / nv),
            Whd=q(wv0[:, 128:]), bq=p["views_linear.0.bias"] + wv0[:, :128] @ p["bottleneck_layer.bias"],
            Wv1=q(p["views_linear.1.weight"]), bv1=p["views_linear.1.bias"], Wrgb=q(p["rgb_layer.weight"]), brgb=p["rgb_layer.bias"],
            bsig=p["density_layer.bias"][0], E=E)

    def project(self, p):
        """Per map: P (nv, H, W, 256) = [P0 | P3] = F . Wsel^T over the map's channels."""
        q = lambda x: r16(x, self.rnd)
        E = 84 if self.is_bg else 63
        w0, w3 = p["pts_linears.0.weight"], p["pts_linears.3.weight"]
        out = []
        for k, fm in enumerate((self.sc.latent, self.sc.planes_xz, self.sc.planes_xy, self.sc.planes_yz)):
            c0 = E + (512 if k else 0)
            C = fm.shape[1]
            wsel = torch.cat([w0[:, c0:c0 + C], w3[:, 128 + c0:128 + c0 + C]], 0)          # (256, C)
            out.append(q(torch.einsum("vchw,nc->vhwn", q(fm), q(wsel))))
        return out

    # ---- stages ----
    def taps(self, gx, gy, H, W):
        """Base texel (x0, y0) (long) and the fp16 weights (..., 4) of nw, ne, sw, se: zero for a tap outside the map."""
        x0, y0, w = orc.bilinear_quad(gx, gy, H, W)
        return x0.long(), y0.long(), r16(w, self.rnd)

    def blend(self, m: int, x0, y0, w, groups=None):
        """sum_taps w . P[tap] for map m: (nv, B, N, 256); an out-of-range tap reads zeros (the TMA window's zero fill)."""
        pm = self.pmaps[m]
        _, H, W, _ = pm.shape
        v = torch.arange(self.nv, device=self.dev).reshape(-1, 1, 1)
        out = 0
        for k, (dx, dy) in enumerate(((0, 0), (1, 0), (0, 1), (1, 1))):
            xx, yy = x0 + dx, y0 + dy
            ok = (xx >= 0) & (xx < W) & (yy >= 0) & (yy < H)
            out = out + pm[v, yy.clamp(0, H - 1), xx.clamp(0, W - 1)] * (w[..., k] * ok)[..., None]
        return out

    def lookups(self, g: Geometry, groups=None):
        """Per map the blended [P0 | P3] rows; `groups` (window_groups of the same geometry) is only used by mutated blends."""
        out = []
        for m, (gx, gy, H, W) in enumerate(g.grids):
            x0, y0, w = self.taps(gx, gy, H, W)
            out.append(self.blend(m, x0, y0, w, None if groups is None else groups[m]))
        return out

    def encode(self, enc_in):
        """Positional encoding, fp16 (exact sin / cos: the kernel's __sinf + double-angle recurrence is not restated)."""
        return r16(orc.pos_enc(enc_in, 0, 10), self.rnd)

    def trunk(self, enc, look: List[Tensor]):
        """h3 (nv, B, N, 128) from the fp16 encoding and the per-map lookups."""
        q = lambda x: r16(x, self.rnd)
        W = self.W
        g0 = sum(a[..., :128] for a in look)
        g3 = sum(a[..., 128:] for a in look)
        h = torch.relu(q(enc @ W["W0enc"].T + W["b0"] + g0))
        h = torch.relu(q(h @ W["W1"].T + W["b1"]))
        h = torch.relu(q(h @ W["W2"].T + W["b2"]))
        return torch.relu(q(enc @ W["W3enc"].T + W["b3"] + g3 + h @ W["W3h"].T))

    def q1_dirs(self, dirs_cam, B, N, chunk):
        """mean over views of the direction encoding of each row's quirk-Q1 conditioning ray, fp16: (B, N, 27)."""
        denc = orc.pos_enc(dirs_cam, 0, 4)                       # (nv, B, 27)
        ch = chunk if chunk > 0 else B
        rows = []
        for c0 in range(0, B, ch):
            Bc = min(ch, B - c0)
            rows.append(orc.q1_dir_tile(denc[:, c0:c0 + Bc], N).reshape(self.nv, Bc, N, -1))
        return r16(torch.cat(rows, 1).mean(0), self.rnd)

    def head(self, h3, dmean):
        q = lambda x: r16(x, self.rnd)
        W = self.W
        hs = h3.sum(0)                                            # sum over views, fp32 in the kernel (never rounded)
        qv = q(torch.relu(hs @ W["Whh"].T + dmean @ W["Whd"].T + W["bq"]))
        v1 = q(torch.relu(qv @ W["Wv1"].T + W["bv1"]))
        rgb = torch.sigmoid(v1 @ W["Wrgb"].T + W["brgb"]) * 1.002 - 0.001
        sigma = F.softplus(hs @ W["wsig"] + W["bsig"] - 1.0, threshold=20.0)
        return rgb, sigma[..., None]

    # ---- the call ----
    def field(self, o, d, vd, far, t, chunk: int = 0, ray_order: Optional[Tensor] = None):
        """rgb (B, N, 3), sigma (B, N, 1) in fp64 for rays o, d, viewdirs vd, far (B,) and t / s (B, N)."""
        f = lambda x: x.to(self.dev, torch.float64)
        o, d, vd, far, t = f(o), f(d), f(vd), f(far), f(t)
        B, N = t.shape
        g = geometry(self.sc, self.is_bg, o, d, vd, far, t)
        groups = self.window_groups(g, ray_order) if self.needs_groups else None
        h3 = self.trunk(self.encode(g.enc_in), self.lookups(g, groups))
        return self.head(h3, self.q1_dirs(g.dirs_cam, B, N, chunk))

    needs_groups = False          # mutations that depend on the window grouping set this

    def window_groups(self, g: Geometry, ray_order: Optional[Tensor] = None):
        return [window_groups(*self.taps(gx, gy, H, W), ray_order) for gx, gy, H, W in g.grids]


def window_groups(x0: Tensor, y0: Tensor, w: Tensor, ray_order: Optional[Tensor] = None) -> Dict[str, Tensor]:
    """The TC kernel's texel-window grouping (field_tc.cu, window warps) applied to one map's tap quads x0, y0, w (nv, B, N).

    A job is 32 rays (slots 32g..32g+31 of `ray_order`) x 2 consecutive samples x 1 view = 64 rows, row = sample_in_pair * 32 + ray.
    A row is live unless it is padding (ray or sample past the batch) or all its tap weights are zero.  The live rows are keyed by
    their 4x4 box of the pitch-3 lattice anchored at the job's minimum base texel; windows are numbered by first appearance in row
    order.  Returns `nwin` (nv, jobs) windows per job, `win` (nv, B, N) each row's window index (-1: not live), `bx`, `by` (nv, B, N)
    the row's base texel offset inside its box, and `job` (nv, B, N) the row's job index."""
    nv, B, N = x0.shape
    dev = x0.device
    order = torch.arange(B, device=dev) if ray_order is None else ray_order.to(dev).long()
    G, SG = (B + TILE_RAYS - 1) // TILE_RAYS, (N + TILE_SAMPLES - 1) // TILE_SAMPLES
    slot = torch.arange(G * TILE_RAYS, device=dev).reshape(G, 1, 1, 1, TILE_RAYS)
    samp = (torch.arange(SG, device=dev).reshape(1, SG, 1, 1, 1) * TILE_SAMPLES
            + torch.arange(2, device=dev).reshape(1, 1, 2, 1, 1) * 2 + torch.arange(2, device=dev).reshape(1, 1, 1, 2, 1))
    slot, samp = torch.broadcast_tensors(slot, samp)                                   # (G, SG, half, pair, 32)
    pad = (slot >= B) | (samp >= N)
    rid = order[slot.clamp(max=B - 1)]
    sid = samp.clamp(max=N - 1)
    J = G * SG * 2
    rid, sid, pad = rid.reshape(J, 64), sid.reshape(J, 64), pad.reshape(J, 64)
    X, Y = x0[:, rid, sid], y0[:, rid, sid]                                            # (nv, J, 64)
    live = (w[:, rid, sid] != 0).any(-1) & ~pad
    big = torch.iinfo(torch.long).max
    xm = torch.where(live, X, big).min(-1, keepdim=True).values
    ym = torch.where(live, Y, big).min(-1, keepdim=True).values
    kx, ky = torch.where(live, X - xm, 0) // PITCH, torch.where(live, Y - ym, 0) // PITCH
    same = (kx[..., :, None] == kx[..., None, :]) & (ky[..., :, None] == ky[..., None, :]) & live[..., None, :] & live[..., :, None]
    first = same.int().argmax(-1)                                                      # first row with the same box
    isfirst = live & (first == torch.arange(64, device=dev))
    rank = torch.cumsum(isfirst.long(), -1) - 1
    win = torch.where(live, rank.gather(-1, first), -1)
    out = {"nwin": isfirst.sum(-1)}
    # scatter the per-row values back to (nv, B, N); padding rows are dropped
    keep = ~pad
    r, s = rid[keep], sid[keep]
    jidx = torch.arange(J, device=dev).reshape(J, 1).expand(J, 64)[keep]
    for name, val in (("win", win), ("bx", X - xm - PITCH * kx), ("by", Y - ym - PITCH * ky)):
        o = torch.full((nv, B, N), -1, dtype=torch.long, device=dev)
        o[:, r, s] = torch.where(live, val, -1)[:, keep]
        out[name] = o
    jb = torch.full((B, N), -1, dtype=torch.long, device=dev)
    jb[r, s] = jidx
    out["job"] = jb.expand(nv, B, N)
    return out
