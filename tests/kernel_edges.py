"""Constructed edge cases for the composite and binning kernels, and a plain float64 reference of the composite.

`composite_ref64` restates the per-tile front-to-back composite (App. A.6 as the oracle documents it) in torch float64,
vectorised over (pixel x list entry) per tile, and takes its gradients from autograd with the skip / termination masks
computed once and then held fixed.  It shares no code with the oracle (oracle.c) or the kernels, so it checks the
oracle's re-associated backward algebra (`S / (1 - aG)`) independently.

The case builders return hand-built tile lists (`ids/start/end`), so every list length and termination point is exactly
what the case claims; `tests/test_kernel_edges_cpu.py` checks those claims with the fp64 reference.  Pixel sizes are
powers of two and principal points multiples of 1/4 pixel, so every pixel position `tl + g * ps` is exact in fp32 and all
implementations evaluate the same positions.
"""
from __future__ import annotations

import math

import numpy as np
import torch

TILE = 16
KMIN = float(np.float32(1.0 / 255.0))  # kMinRenderAlpha (fp32 constant)
ACLAMP = float(np.float32(0.99))       # alpha clamp (fp32 constant)
PS = 1.0 / 128.0                       # pixel size in camera-plane units
BATCHES = (32, 64, 128, 256)           # staged batch sizes of the composite kernels
EPS32 = 2.0 ** -24
THRESHES = (0.0, 1e-4, 0.5, 1.0, 1.5)
GEOMETRIES = ((1, 1), (5, 37), (16, 17), (17, 16), (33, 250), (105, 162), (210, 324))
KINDS = ("rgb", "scalar", "sh1", "sh1bg", "sh2", "sh2bg", "sh3", "sh3bg", "sh4", "sh4bg")


def lengths_for(B):
    return (1, 31, 32, 33, B - 1, B, B + 1, 2 * B - 1, 2 * B, 2 * B + 1, 3 * B + 5)


LENGTHS = tuple(sorted({n for B in BATCHES for n in lengths_for(B)}))


# ------------------------------------------------------------------------------------------------------------------
# float64 reference
# ------------------------------------------------------------------------------------------------------------------
def pixel_positions(topleft, psx, psy, gx, gy):
    """fp32 pixel-corner positions tl + g*ps, rounded once (the kernels' fmaf), as float64"""
    tl = topleft.double()
    px = (tl[0] + gx.double() * float(np.float32(psx))).float().double()
    py = (tl[1] + gy.double() * float(np.float32(psy))).float().double()
    return px, py


def sh_basis64(d, C):
    """[P,3] unit directions -> [P,C*C] real SH basis (gsb200_math.cuh sh_basis, in float64)"""
    x, y, z = d[:, 0], d[:, 1], d[:, 2]
    xy, xz, yz, x2, y2, z2 = x * y, x * z, y * z, x * x, y * y, z * z
    Y = [torch.full_like(x, 0.28209479177387814)]
    if C > 1:
        Y += [-0.48860251190291987 * y, 0.48860251190291987 * z, -0.48860251190291987 * x]
    if C > 2:
        Y += [1.0925484305920792 * xy, -1.0925484305920792 * yz, 0.94617469575755997 * z2 - 0.31539156525251999,
              -1.0925484305920792 * xz, 0.54627421529603959 * x2 - 0.54627421529603959 * y2]
    if C > 3:
        Y += [0.59004358992664352 * y * (-3.0 * x2 + y2), 2.8906114426405538 * xy * z,
              0.45704579946446572 * y * (1.0 - 5.0 * z2), 0.3731763325901154 * z * (5.0 * z2 - 3.0),
              0.45704579946446572 * x * (1.0 - 5.0 * z2), 1.4453057213202769 * z * (x2 - y2),
              0.59004358992664352 * x * (-x2 + 3.0 * y2)]
    return torch.stack(Y, dim=-1)


def pixel_dir64(px, py, c2w9):
    """normalize(rows(c2w9) . (px, py, 1)) (gsb200_math.cuh pixel_dir) in float64"""
    R = c2w9.reshape(-1)[:9].double().view(3, 3)
    p = torch.stack([px, py, torch.ones_like(px)], dim=-1)
    d = p @ R.T
    return d / d.norm(dim=-1, keepdim=True)


def composite_ref64(*args, **kw):
    # many small ops per tile: more than a few intra-op threads only add scheduling overhead
    n = torch.get_num_threads()
    torch.set_num_threads(min(n, 4))
    try:
        return _composite_ref64(*args, **kw)
    finally:
        torch.set_num_threads(n)


def _composite_ref64(mean2d, cov2d, payload, alpha, start, end, ids, topleft, psx, psy, H, W, thresh, *, kind="rgb",
                     bg=None, c2w9=None, C=None, bg_rgb=None, gout=None, keep_masks=False):
    """The per-tile composite in float64.

    kind "rgb": payload [N,3], out = sum w*color + T*bg (bg [H,W,3] or None);  "scalar": payload [N];
    "sh": payload [N,3,C*C], colour sigmoid(sum_k sh[c,k] Y_k(dir)), out += T*bg_rgb when given.
    Per pixel, entry i is evaluated while T >= thresh (checked before it), skipped when a*G < 1/255 (a = min(alpha, 0.99),
    G = exp(-q/2) with the reference's q), otherwise blended: w = a*G*T, T *= 1 - a*G.
    Returns a dict: out, T, margin (min |a*G*255 - 1| over evaluated pairs), term_margin (min |T - thresh| / thresh over
    the values T took), stop (entries evaluated), and with `gout` the gradients of sum(out * gout) w.r.t. mean2d, cov2d,
    payload, alpha (+ bg).  The alpha clamp is straight-through (the reference's g_alpha has no clamp gate)."""
    N = mean2d.shape[0]
    want_grad = gout is not None
    leaf = lambda t: t.detach().double().clone().requires_grad_(want_grad)
    m, cv, al = leaf(mean2d.reshape(N, 2)), leaf(cov2d.reshape(N, 4)), leaf(alpha.reshape(N))
    pay = leaf(payload)
    bgt = leaf(bg) if (bg is not None and kind == "rgb") else None
    a_all = al - (al - al.clamp(max=ACLAMP)).detach()
    nch = 1 if kind == "scalar" else 3
    th_ = float(thresh)
    pix_list, val_list, T_list = [], [], []
    out_T = torch.ones(H * W, dtype=torch.float64)
    margin = torch.full((H * W,), math.inf, dtype=torch.float64)
    term = torch.full((H * W,), math.inf, dtype=torch.float64)
    stop = torch.zeros(H * W, dtype=torch.int64)
    masks = {}
    n_tiles_h, n_tiles_w = (H + TILE - 1) // TILE, (W + TILE - 1) // TILE
    start, end, ids = start.cpu(), end.cpu(), ids.cpu()
    for tile in range(n_tiles_h * n_tiles_w):
        s = int(start[tile])
        n = 0 if s < 0 else int(end[tile]) - s
        if n <= 0:
            continue
        ty, tx = divmod(tile, n_tiles_w)
        ly, lx = torch.meshgrid(torch.arange(TILE), torch.arange(TILE), indexing="ij")
        gy, gx = (ty * TILE + ly).reshape(-1), (tx * TILE + lx).reshape(-1)
        inside = (gy < H) & (gx < W)
        loc = torch.nonzero(inside).squeeze(1)  # local pixel index ly*16+lx
        gy, gx = gy[inside], gx[inside]
        pidx = gy * W + gx
        px, py = pixel_positions(topleft, psx, psy, gx, gy)
        idx = ids[s:s + n].long()
        mm, c, a = m[idx], cv[idx], a_all[idx]
        dx, dy = px[:, None] - mm[None, :, 0], py[:, None] - mm[None, :, 1]
        c0, c1, c2, c3 = c[:, 0], c[:, 1], c[:, 2], c[:, 3]
        q = ((dx * c3 - dy * c2) * dx + (-dx * c1 + dy * c0) * dy) / (c0 * c3 - c1 * c2)
        G = torch.exp(-0.5 * q)
        aG = a[None, :] * G
        with torch.no_grad():
            aGd = aG.detach()
            pas = aGd >= KMIN
            f = torch.where(pas, 1.0 - aGd, torch.ones_like(aGd))
            Ta = torch.cumprod(f, dim=1)
            Tb = torch.cat([torch.ones_like(Ta[:, :1]), Ta[:, :-1]], dim=1)
            ev = Tb >= th_
            bl = ev & pas
            stop[pidx] = ev.sum(1)
            mg = torch.where(ev, (aGd * 255.0 - 1.0).abs(), torch.full_like(aGd, math.inf))
            margin[pidx] = mg.amin(1)
            if th_ > 0:
                tm = torch.where(bl, (Ta - th_).abs() / th_, torch.full_like(Ta, math.inf))
                term[pidx] = tm.amin(1)
        if keep_masks:
            full = torch.zeros(TILE * TILE, n, dtype=torch.bool)
            full[loc] = bl
            masks[tile] = full
        fct = torch.where(bl, 1.0 - aG, torch.ones_like(aG))
        Tc = torch.cumprod(fct, dim=1)
        Tbg = torch.cat([torch.ones_like(Tc[:, :1]), Tc[:, :-1]], dim=1)
        w = torch.where(bl, aG * Tbg, torch.zeros_like(aG))
        Tfin = Tc[:, -1]
        if kind == "rgb":
            val = w @ pay[idx]
            if bgt is not None:
                val = val + Tfin[:, None] * bgt.reshape(H * W, 3)[pidx]
        elif kind == "scalar":
            val = (w @ pay.reshape(-1)[idx])[:, None]
        else:
            Y = sh_basis64(pixel_dir64(px, py, c2w9), C)
            col = torch.sigmoid(torch.einsum("pk,nck->pnc", Y, pay[idx]))
            val = (w[:, :, None] * col).sum(1)
            if bg_rgb is not None:
                val = val + Tfin[:, None] * bg_rgb.double()[None, :]
        pix_list.append(pidx)
        val_list.append(val)
        T_list.append(Tfin)
        out_T[pidx] = Tfin.detach()
    # empty tiles keep T = 1: RGB shows the background there, SH with a background writes it
    base = torch.zeros(H * W, nch, dtype=torch.float64)
    if kind == "rgb" and bgt is not None:
        base = base + bgt.reshape(H * W, 3)
    if kind.startswith("sh") and bg_rgb is not None:
        base = base + bg_rgb.double()[None, :]
    if pix_list:
        P = torch.cat(pix_list)
        out = base.index_put((P,), torch.cat(val_list))
    else:
        out = base
    res = dict(out=out.reshape(H, W, nch) if nch == 3 else out.reshape(H, W), T=out_T.reshape(H, W),
               margin=margin.reshape(H, W), term_margin=term.reshape(H, W), stop=stop.reshape(H, W))
    if keep_masks:
        res["masks"] = masks
    if want_grad:
        loss = (out.reshape(-1) * gout.detach().double().reshape(-1)).sum()
        ins = [m, cv, pay, al] + ([bgt] if bgt is not None else [])
        gr = torch.autograd.grad(loss, ins, allow_unused=True)
        z = lambda g_, t: torch.zeros_like(t) if g_ is None else g_
        res.update(g_mean2d=z(gr[0], m), g_cov2d=z(gr[1], cv).view(N, 2, 2), g_pay=z(gr[2], pay),
                   g_alpha=z(gr[3], al))
        if bgt is not None:
            res["g_bg"] = z(gr[4], bgt)
        res["out"] = res["out"].detach()
    return res


def flip_free(ref, tol=1e-5):
    """pixels where fp32 and fp64 cannot legitimately take different branches: threshold and termination margins >= tol"""
    return (ref["margin"] >= tol) & (ref["term_margin"] >= tol)


def kernel_aG_error(case, px, py, gidx):
    """Forward-error bound of the kernels' fp32 a*G for pair (pixel, Gaussian gidx): they evaluate
    G = exp2(-(u^2+v^2)), u = p0*dx + p1*dy, v = p2*dy, from the fp32 Cholesky factor of the conic (make_splat).  For a
    splat with axis ratio r the sum u cancels and its error grows ~ r * eps; the bound is the standard one of that
    expression (4 roundings in u, 3 in v, 2 in the sum of squares) plus ex2.approx's 2^-22 relative error."""
    c = case["cov2d"].reshape(-1, 4)[gidx].double()
    c0, c1, c2, c3 = (float(v) for v in c)
    det = c0 * c3 - c1 * c2
    A, B, Cc = c3 / det, -0.5 * (c1 + c2) / det, c0 / det
    l00 = math.sqrt(A)
    l01 = B / l00
    s = 0.84932180028801907
    p0, p1, p2 = (float(np.float32(s * l00)), float(np.float32(s * l01)), float(np.float32(s * math.sqrt(Cc - l01 * l01))))
    mx, my = (float(v) for v in case["mean2d"][gidx].double())
    dx, dy = px - mx, py - my
    u, v = p0 * dx + p1 * dy, p2 * dy
    s1, s2 = (p0 * dx).abs() + (p1 * dy).abs(), (p2 * dy).abs()
    de = EPS32 * (8.0 * u.abs() * s1 + 6.0 * v.abs() * s2 + 2.0 * (u * u + v * v))
    a = min(float(case["alpha"][gidx]), ACLAMP)
    aG = a * torch.exp2(-(u * u + v * v))
    return aG * (math.log(2.0) * de + 2.0 ** -21 + 4 * EPS32)


# ------------------------------------------------------------------------------------------------------------------
# case builders
# ------------------------------------------------------------------------------------------------------------------
class _Builder:
    """Gaussians in pixel units on a camera plane with pixel size PS; tile lists by hand."""

    def __init__(self, name, H, W, seed, cx=None, cy=None):
        self.name, self.H, self.W = name, H, W
        self.g = np.random.default_rng(seed)
        self.cx = (W / 2.0) if cx is None else cx
        self.cy = (H / 2.0) if cy is None else cy
        self.th, self.tw = (H + TILE - 1) // TILE, (W + TILE - 1) // TILE
        self.mean, self.cov, self.alpha = [], [], []
        self.lists = {}

    def add(self, x, y, sx, sy, theta, alpha):
        """a Gaussian centred at pixel coordinates (x, y), std devs (sx, sy) px along axes rotated by theta"""
        R = np.array([[math.cos(theta), -math.sin(theta)], [math.sin(theta), math.cos(theta)]])
        S = R @ np.diag([sx * sx, sy * sy]) @ R.T * (PS * PS)
        return self.add_cov(x, y, S, alpha)

    def add_cov(self, x, y, S, alpha):
        self.mean.append([(x - self.cx) * PS, (y - self.cy) * PS])
        c = np.float32([S[0, 0], S[0, 1], S[0, 1], S[1, 1]])  # c1 == c2 bit for bit
        self.cov.append(c)
        self.alpha.append(alpha)
        return len(self.mean) - 1

    def push(self, tile, gid):
        self.lists.setdefault(tile, []).append(gid)

    def build(self, thresh=1e-4, **meta):
        N = len(self.mean)
        g = torch.Generator().manual_seed(int(self.g.integers(1 << 30)))
        ids, start, end = [], -torch.ones(self.th * self.tw, dtype=torch.int32), -torch.ones(self.th * self.tw,
                                                                                                dtype=torch.int32)
        for t in range(self.th * self.tw):
            lst = self.lists.get(t, [])
            if lst:
                start[t] = len(ids)
                ids += lst
                end[t] = len(ids)
        ang = 0.35
        R = torch.tensor([[math.cos(ang), 0.0, math.sin(ang)], [0.0, 1.0, 0.0], [-math.sin(ang), 0.0, math.cos(ang)]])
        R = R @ torch.tensor([[1.0, 0.0, 0.0], [0.0, math.cos(0.2), -math.sin(0.2)], [0.0, math.sin(0.2), math.cos(0.2)]])
        case = dict(
            name=self.name, H=self.H, W=self.W, n_tiles_h=self.th, n_tiles_w=self.tw, psx=PS, psy=PS, thresh=thresh,
            topleft=torch.tensor([-self.cx * PS, -self.cy * PS], dtype=torch.float32),
            mean2d=torch.tensor(np.float32(self.mean)).reshape(N, 2),
            cov2d=torch.tensor(np.float32(self.cov)).reshape(N, 2, 2),
            alpha=torch.tensor(np.float32(self.alpha)).reshape(N),
            color=torch.rand(N, 3, generator=g), scalar=0.5 + 1.5 * torch.rand(N, generator=g),
            sh=(0.5 * torch.randn(N, 3, 16, generator=g)),
            ids=torch.tensor(ids, dtype=torch.int32), start=start, end=end,
            c2w9=torch.cat([R.reshape(-1), torch.tensor([0.1, -0.2, 2.5])]).float(),
            bg=torch.rand(self.H, self.W, 3, generator=g), bg_rgb=torch.tensor([0.2, 0.5, 0.7]),
            gout=torch.randn(self.H, self.W, 3, generator=g), meta=meta)
        return case


def _filler(b, tile, rng, x0=-2.0, x1=18.0, y0=-2.0, y1=18.0, a=(0.02, 0.15), s=(1.0, 3.0)):
    tx, ty = tile % b.tw, tile // b.tw
    sx = rng.uniform(*s)
    return b.add(tx * TILE + rng.uniform(x0, x1), ty * TILE + rng.uniform(y0, y1), sx, sx / rng.uniform(1.0, 3.0),
                 rng.uniform(0, math.pi), rng.uniform(*a))


def lengths_case(thresh=1e-4, seed=1):
    """one tile per list length n in LENGTHS (1, 31, 32, 33, B-1, B, B+1, 2B-1, 2B, 2B+1, 3B+5 for every batch size B):
    small low-alpha Gaussians spread over the tile, so every warp has hits."""
    tw = 5
    th = (len(LENGTHS) + tw - 1) // tw
    b = _Builder(f"lengths_t{thresh:g}", th * TILE, tw * TILE, seed)
    for t, n in enumerate(LENGTHS):
        for _ in range(n):
            b.push(t, _filler(b, t, b.g))
    return b.build(thresh, lengths={t: n for t, n in enumerate(LENGTHS)})


def termination_case(thresh=1e-4, seed=2):
    """one tile per batch size B, list length 3B+5.  Two tile-wide near-opaque layers (alpha 1.0 -> clamped, then 0.987)
    at entries B-3, B-2 leave T ~ 1.3e-4; then a "kicker" per 4-pixel row of warps (alpha 1.0, sigma_y = 1 px, tile wide)
    at entry s_row in {B-1, B, B+1, B+B/2} takes that row below 1e-4 and leaves the rows next to it above.  So at
    thresh = 1e-4 the two warps of a row evaluate exactly s_row + 1 entries, different rows of one CTA stop in different
    batches, one inside the batch that was prefetched.  Every other entry is a faint filler centred in a random warp
    block (alpha just above 1/255), which makes the hit count of each warp at its last batch vary mod 4."""
    b = _Builder(f"termination_t{thresh:g}", 2 * TILE, 2 * TILE, seed)
    stops = {}
    for t, B in enumerate(BATCHES):
        tx, ty = t % 2, t // 2
        n = 3 * B + 5
        targets = [B - 1, B, B + 1, B + B // 2]
        order = b.g.permutation(4)
        rows = {targets[k]: int(r) for k, r in zip(range(4), order)}
        for j in range(n):
            if j == B - 3:
                gid = b.add(tx * TILE + 7.5, ty * TILE + 7.5, 2000.0, 2000.0, 0.0, 1.0)
            elif j == B - 2:
                gid = b.add(tx * TILE + 7.5, ty * TILE + 7.5, 2000.0, 2000.0, 0.0, 0.9868)
            elif j in rows:
                r = rows[j]
                gid = b.add(tx * TILE + 7.5, ty * TILE + 4 * r + 1.5, 2000.0, 1.0, 0.0, 1.0)
                stops[(t, r)] = j + 1
            else:
                w = int(b.g.integers(8))
                bx, by = tx * TILE + (w & 1) * 8, ty * TILE + (w >> 1) * 4
                sg = b.g.uniform(0.7, 1.2)
                gid = b.add(bx + b.g.uniform(0.5, 6.5), by + b.g.uniform(0.5, 2.5), sg, sg, 0.0, b.g.uniform(0.0042, 0.006))
            b.push(t, gid)
    return b.build(thresh, stops=stops, batches={t: B for t, B in enumerate(BATCHES)})


def geometry_case(H, W, thresh=1e-4, seed=3):
    """random Gaussians (some centred outside the image) binned by their 3-sigma box clamped to the image: partial
    tiles, warps entirely outside the image, H % 4 != 0, non-square grids, an off-centre principal point, and (when the
    grid has more than 3 tiles) one empty tile."""
    b = _Builder(f"geometry_{H}x{W}", H, W, seed + H * 1000 + W, cx=0.25 * round(4 * (0.37 * W + 3.3)),
                 cy=0.25 * round(4 * (0.61 * H - 1.7)))
    N = max(6, H * W // 30)
    order = b.g.permutation(N)  # depth order
    recs = []
    for _ in range(N):
        x, y = b.g.uniform(-6, W + 6), b.g.uniform(-6, H + 6)
        sx = b.g.uniform(0.6, 5.0)
        sy = sx / b.g.uniform(1.0, 4.0)
        gid = b.add(x, y, sx, sy, b.g.uniform(0, math.pi), b.g.uniform(0.05, 0.95))
        r = 3.0 * sx + 1.0
        x0, x1 = max(0, int((x - r) // TILE)), min(b.tw - 1, int((x + r) // TILE))
        y0, y1 = max(0, int((y - r) // TILE)), min(b.th - 1, int((y + r) // TILE))
        recs.append((gid, x0, x1, y0, y1))
    empty = 1 if b.th * b.tw > 3 else -1
    for k in order:
        gid, x0, x1, y0, y1 = recs[k]
        for ty in range(y0, y1 + 1):
            for tx in range(x0, x1 + 1):
                if ty * b.tw + tx != empty:
                    b.push(ty * b.tw + tx, gid)
    return b.build(thresh, empty_tile=empty)


GRAZE_ALPHAS = (KMIN * 1.02, 0.05, 0.5, 0.99, 1.0)


def grazing_case(seed=4):
    """8 x 8 tiles, each with a one-entry list: one Gaussian (random rotation, axis ratio up to 10^3, alpha in
    GRAZE_ALPHAS) scaled so that its a*G = 1/255 ellipse just reaches the nearest pixel of a chosen warp block, from
    inside (that pixel is blended by a relative margin of 3e-5 .. 3e-3 in a*G*255) or from outside (it is skipped by
    that margin).  The centre lies beyond a corner, beyond an edge, or inside the block, up to 30 px away: outside the
    tile and, for border tiles, outside the image."""
    b = _Builder("grazing", 128, 128, seed, cx=61.25, cy=66.75)
    targets = {}
    for t in range(b.th * b.tw):
        kind = ("corner", "edge", "inside")[t % 3]
        a = GRAZE_ALPHAS[(t // 3) % len(GRAZE_ALPHAS)]
        inside = bool((t // 15) % 2)
        for _ in range(500):  # fp32 rounding moves a thin conic by ~eps * ratio^2: keep a draw whose rounded inputs land
            g = _graze_draw(b, t, kind, a, inside)
            if g is not None:
                break
        assert g is not None, t
        x, y, S, w, mt, ratio = g
        b.push(t, b.add_cov(x, y, S, a))
        targets[t] = dict(warp=w, kind=kind, inside=inside, margin=mt, ratio=ratio, alpha=a)
    return b.build(1e-4, targets=targets)


def _graze_draw(b, t, kind, a, inside):
    rng = b.g
    tx, ty = t % b.tw, t // b.tw
    w = int(rng.integers(8))
    bx, by = tx * TILE + (w & 1) * 8, ty * TILE + (w >> 1) * 4
    ratio = 10.0 ** rng.uniform(0, 3) if kind != "inside" else 10.0 ** rng.uniform(0, 1)
    th_ = rng.uniform(0, math.pi)
    dist = 10.0 ** rng.uniform(-0.3, 1.5)
    if kind == "corner":
        sx, sy = (-1, 1)[rng.integers(2)], (-1, 1)[rng.integers(2)]
        x = bx + (7 if sx > 0 else 0) + sx * (0.5 + dist * rng.uniform(0.2, 1))
        y = by + (3 if sy > 0 else 0) + sy * (0.5 + dist * rng.uniform(0.2, 1))
    elif kind == "edge":
        side = int(rng.integers(4))
        if side < 2:
            x, y = (bx - 0.5 - dist, bx + 7.5 + dist)[side], by + rng.uniform(0, 3)
        else:
            x, y = bx + rng.uniform(0, 7), (by - 0.5 - dist, by + 3.5 + dist)[side - 2]
    else:
        x, y = bx + int(rng.integers(7)) + 0.5 + rng.uniform(-0.1, 0.1), by + int(rng.integers(3)) + 0.5
    R = np.array([[math.cos(th_), -math.sin(th_)], [math.sin(th_), math.cos(th_)]])
    S0 = R @ np.diag([1.0, 1.0 / ratio ** 2]) @ R.T
    gx, gy = np.meshgrid(np.arange(bx, bx + 8), np.arange(by, by + 4))
    d = np.stack([gx.ravel() - x, gy.ravel() - y], 1)
    q = np.einsum("pi,ij,pj->p", d, np.linalg.inv(S0), d)
    aa = min(float(np.float32(a)), ACLAMP)
    q0 = 2.0 * math.log(255.0 * aa)
    mt = 10.0 ** rng.uniform(math.log10(3e-5), math.log10(3e-3))
    qt = q0 + (-2.0 if inside else 2.0) * mt  # a*G*255 = exp((q0 - q)/2) ~ 1 +/- mt
    S = S0 * (q.min() / qt) * PS * PS  # q scales as 1/s when S0 does as s
    # what the fp32 inputs give, in float64: camera-plane positions and the reference's q
    c = np.float64(np.float32([S[0, 0], S[0, 1], S[1, 1]]))
    mx, my = np.float64(np.float32((x - b.cx) * PS)), np.float64(np.float32((y - b.cy) * PS))
    px = np.float64(np.float32(-b.cx * PS + gx.ravel() * PS)) - mx
    py = np.float64(np.float32(-b.cy * PS + gy.ravel() * PS)) - my
    det = c[0] * c[2] - c[1] * c[1]
    if not det > 0:
        return None
    qr = ((px * c[2] - py * c[1]) * px + (-px * c[1] + py * c[0]) * py) / det
    aG = aa * np.exp(-0.5 * qr)
    m = np.abs(aG * 255.0 - 1.0)
    k = int(np.argmin(m))
    if not (3e-5 <= m[k] <= 3e-3) or (aG[k] >= KMIN) != inside or (aG > KMIN * (1 + 3e-3)).any():
        return None
    return x, y, S, w, float(m[k]), ratio


def degenerate_case(seed=5):
    """two tiles.  Tile 0 lists only covariances with det <= 0 or c0 <= 0 and Gaussians with NaN alpha; tile 1 lists
    the same kinds interleaved with ordinary Gaussians (meta["valid"] marks the ordinary ones).  The library's convention
    is that such entries contribute nothing."""
    b = _Builder("degenerate", 16, 32, seed)
    bad, valid = [], []
    for t in range(2):
        for k in range(12):
            x, y = t * TILE + b.g.uniform(2, 14), b.g.uniform(2, 14)
            s2 = (b.g.uniform(1.5, 4) * PS) ** 2
            kind = k % 4
            if kind == 0:    # det == 0 (rank one)
                S = np.array([[s2, s2], [s2, s2]])
                gid = b.add_cov(x, y, S, 0.8)
            elif kind == 1:  # det < 0
                S = np.array([[s2, 2 * s2], [2 * s2, s2]])
                gid = b.add_cov(x, y, S, 0.8)
            elif kind == 2:  # c0 <= 0 with det > 0 (negative definite) or c0 == 0
                S = np.array([[-s2, 0.0], [0.0, -s2]]) if k % 8 == 2 else np.array([[0.0, 0.0], [0.0, s2]])
                gid = b.add_cov(x, y, S, 0.8)
            else:            # NaN alpha
                gid = b.add(x, y, 2.0, 2.0, 0.0, float("nan"))
            b.push(t, gid)
            bad.append(gid)
            if t == 1:
                gid = b.add(x + 1.0, y - 1.0, b.g.uniform(1, 3), b.g.uniform(1, 3), b.g.uniform(0, 3), b.g.uniform(0.1, 0.9))
                b.push(t, gid)
                valid.append(gid)
    return b.build(1e-4, bad=bad, valid=valid)


# ------------------------------------------------------------------------------------------------------------------
# binning cases: synthetic tile rectangles and depths, no image
# ------------------------------------------------------------------------------------------------------------------
BIN_GRIDS = {  # name -> (tiles_h, tiles_w, N)
    "T65535": (255, 257, 1000),     # largest 16-bit grid; T + 1 = 65536 (async padding still fits 16 bits)
    "T65536": (256, 256, 33),       # 16-bit keys synchronously, 32-bit with the padding key
    "T65538": (2, 32769, 1000),     # 32-bit keys (65 537 is prime: its only grid, 1 x 65 537, exceeds 65 535 tiles a side)
    "T90000": (300, 300, 1000),
    "N1": (256, 257, 1),
    "N31": (300, 300, 31),
    "N32": (255, 257, 32),
}


def binning_case(name, seed=6):
    """tl / br in tiles, depth: Gaussian 0 covers the whole grid (N > 1), one in every 8 (a different lane of every warp
    of 32) has an empty rectangle, depths repeat, include negatives, +0.0 and -0.0."""
    th, tw, N = BIN_GRIDS[name]
    rng = np.random.default_rng(seed + N + th)
    tl = np.zeros((N, 2), np.int32)
    br = np.zeros((N, 2), np.int32)
    for i in range(N):
        w, h = int(rng.integers(1, 5)), int(rng.integers(1, 5))
        x0, y0 = int(rng.integers(0, max(1, tw - w + 1))), int(rng.integers(0, max(1, th - h + 1)))
        tl[i] = (x0, y0)
        br[i] = (min(tw - 1, x0 + w - 1), min(th - 1, y0 + h - 1))
        if i % 8 == (i // 32) % 8:  # zero-count entries, one per 8 lanes, in every warp
            ax = int(rng.integers(2))
            br[i, ax] = tl[i, ax] - 1
    if N > 1:
        tl[0], br[0] = (0, 0), (tw - 1, th - 1)
    pool = np.float32([1.5, 1.5, 2.0, -0.5, -3.0, 0.0, -0.0, 0.25, 7.0, 1e-30, -1e-30])
    depth = np.where(rng.random(N) < 0.5, pool[rng.integers(len(pool), size=N)],
                     np.float32(rng.normal(size=N) * 3)).astype(np.float32)
    if N >= 4:
        depth[1], depth[2] = np.float32(0.0), np.float32(-0.0)
    tl_t, br_t = torch.from_numpy(tl), torch.from_numpy(br)
    cnt = ((br_t - tl_t + 1).clamp(min=0)).prod(dim=1)
    return dict(name=name, n_tiles_h=th, n_tiles_w=tw, tl=tl_t, br=br_t, depth=torch.from_numpy(depth).view(N, 1),
                D=int(cnt.sum()), counts=cnt)
