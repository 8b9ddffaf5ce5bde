"""-m gpu: libgsb200.so against the UNMODIFIED reference `_gs` CUDA extension, same tensors.

Where `oracle/_ref/_gs.so` has been built (oracle/build_ref.sh, from the reference's sources) the two run side by side
on the same B200 and every output is compared whole; elsewhere the comparison runs against a fixed sample of the
extension's outputs recorded that way (tests/golden/ref_c1.npz, ref_c2.npz; tests/util.py::RefGolden)."""
import pytest
import torch

from gsgen_b200.scenes import make_scene
from tests.util import RefGolden, load_ref_ext, ocam_of

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def ref_gs():
    return load_ref_ext()


def _prep_gpu(sc, cam, c2w):
    """cull (ours, checked against the reference separately) + our projection + our AABB count."""
    from gsgen_b200.backend import _backend
    from gsgen_b200.culling import tile_culling_aabb_count
    from gsgen_b200.renderer import project_gaussians

    normals, pts = cam.get_frustum(c2w)
    mask = torch.zeros(sc.N, dtype=torch.bool, device=DEV)
    _backend.culling_gaussian_bsphere(sc.mean, sc.qvec, sc.svec, normals.to(DEV), pts.to(DEV), mask, 6.0)
    m, q, s = sc.mean[mask].contiguous(), sc.qvec[mask].contiguous(), sc.svec[mask].contiguous()
    mean2d, cov2d, _, depth = project_gaussians(m, q, s, c2w, True)
    D, tl, br = tile_culling_aabb_count(mean2d, cov2d, 16, cam, 6.0)
    return mask, mean2d.contiguous(), cov2d.contiguous(), depth.contiguous(), D, tl, br, normals.to(DEV), pts.to(DEV)


@pytest.mark.parametrize("cfg", ["c1", "c2"])
def test_against_reference_extension(ref_gs, oracle_mod, cfg):
    from gsgen_b200.backend import _backend

    R = RefGolden(f"ref_{cfg}", ref_gs)
    live = R.live
    sc = (make_scene("c1") if cfg == "c1" else make_scene("c2")).to(DEV)  # BASELINE configs 1 and 2, full size
    cam, c2w = sc.cams[0], sc.c2ws[0]
    H, W = cam.h, cam.w
    th, tw = cam.n_tiles
    mask, m2, c2, dp, D, tl, br, normals, pts = _prep_gpu(sc, cam, c2w)
    # K1
    rmask = None
    if live:
        rmask = torch.zeros(sc.N, dtype=torch.bool, device=DEV)
        ref_gs.culling_gaussian_bsphere(sc.mean, sc.qvec, sc.svec, normals, pts, rmask, 6.0)
    R.equal("mask", mask, rmask)
    al, col = sc.alpha[mask].contiguous(), sc.color[mask].contiguous()
    # K2-K4 (no exact depth ties in these scenes except c2's padding... identical keys only if equal depth bits)
    mk = lambda: (torch.zeros(D, dtype=torch.int32, device=DEV), -torch.ones(th * tw, dtype=torch.int32, device=DEV),
                  -torch.ones(th * tw, dtype=torch.int32, device=DEV))
    ids, start, end = mk()
    _backend.tile_culling_aabb_start_end(tl, br, ids, start, end, dp, th, tw)
    rids, rstart, rend = mk() if live else (ids, None, None)  # stored: the lists below are ours, pinned here
    if live:
        ref_gs.tile_culling_aabb_start_end(tl, br, rids, rstart, rend, dp, th, tw)
    torch.cuda.synchronize()
    R.equal("start", start, rstart)
    R.equal("end", end, rend)
    R.sorted_ids("ids", ids, dp, rids if live else None)
    topleft = torch.tensor([-cam.cx / cam.fx, -cam.cy / cam.fy], device=DEV)
    psx, psy = 1.0 / cam.fx, 1.0 / cam.fy
    common = (16, th, tw, psx, psy, H, W, 1e-4)
    g = torch.Generator().manual_seed(77)
    gout = torch.randn(H, W, 3, generator=g).to(DEV)
    bg = torch.rand(H, W, 3, generator=g).to(DEV)
    cfg_o = oracle_mod.view_cfg(ocam_of(cam))
    cpu = (m2.cpu(), c2.cpu(), al.cpu(), start.cpu(), end.cpu(), rids.cpu(), topleft.cpu())
    _memo = {}

    def rgb_margin():  # fp64 Gaussian evaluation (RGB and scalar kernels, kernels.h:195-224)
        if "rgb" not in _memo:
            _memo["rgb"] = oracle_mod.composite_rgb_fwd(cpu[0], cpu[1], col.cpu(), cpu[2], cpu[3], cpu[4], cpu[5],
                                                        cpu[6], cfg_o, want_margin=True)[3]
        return _memo["rgb"]

    def close(key, ours, ref, margin_fn=rgb_margin, exact_fn=None):
        # every pixel over 1e-4 must be explained (threshold flip / reference-side fp32 rounding): tests/util.py
        return R.image(key, ours, ref, margin_fn, exact_fn)

    # K5 / K6
    o, T = torch.zeros(H, W, 3, device=DEV), torch.ones(H, W, 1, device=DEV)
    ro, rT = torch.zeros(H, W, 3, device=DEV), torch.ones(H, W, 1, device=DEV)
    _backend.tile_based_vol_rendering_start_end_with_T(m2, c2, col, al, start, end, rids, o, topleft, *common, T)
    if live:
        ref_gs.tile_based_vol_rendering_start_end_with_T(m2, c2, col, al, start, end, rids, ro, topleft, *common, rT)
    torch.cuda.synchronize()
    close("rgb", o, ro)
    close("T", T.view(H, W), rT.view(H, W))
    # the backward reads the forward's output: the reference's where it ran, else ours (pinned just above)
    final = ((ro + rT * bg) if live else (o + T * bg)).contiguous()
    gz = lambda: (torch.zeros_like(m2), torch.zeros_like(c2), torch.zeros_like(col), torch.zeros_like(al))
    gm, gc, gcol, ga = gz()
    rgm, rgc, rgcol, rga = gz()
    _backend.tile_based_vol_rendering_backward_start_end(m2, c2, col, al, start, end, rids, final, gm, gc, gcol, ga,
                                                         gout, topleft, *common)
    if live:
        ref_gs.tile_based_vol_rendering_backward_start_end(m2, c2, col, al, start, end, rids, final, rgm, rgc, rgcol,
                                                           rga, gout, topleft, *common)
    torch.cuda.synchronize()
    for a_, b_, n_ in ((gm, rgm, "g_mean2d"), (gc, rgc, "g_cov2d"), (gcol, rgcol, "g_color"), (ga, rga, "g_alpha")):
        R.grad(n_, a_, b_)
    # K7 / K8 with the depth payload
    so, sT = torch.zeros(H * W, device=DEV), torch.ones(H, W, 1, device=DEV)
    rso, rsT = torch.zeros(H * W, device=DEV), torch.ones(H, W, 1, device=DEV)
    _backend.tile_based_vol_rendering_scalar(m2, c2, dp, al, start, end, rids, so, topleft, *common, sT)
    if live:
        ref_gs.tile_based_vol_rendering_scalar(m2, c2, dp, al, start, end, rids, rso, topleft, *common, rsT)
    torch.cuda.synchronize()
    zs = R.scalar("depth_scale", lambda: max(1.0, float(rso.abs().max())))
    close("depth image", so.view(H, W) / zs, rso.view(H, W) / zs)
    gso = gout[..., 0].contiguous().view(-1)
    gm, gc, gs_, ga = torch.zeros_like(m2), torch.zeros_like(c2), torch.zeros_like(dp), torch.zeros_like(al)
    rgm, rgc, rgs, rga = torch.zeros_like(m2), torch.zeros_like(c2), torch.zeros_like(dp), torch.zeros_like(al)
    _backend.tile_based_vol_rendering_scalar_backward(m2, c2, dp, al, start, end, rids, rso if live else so, gm, gc, gs_,
                                                      ga, gso, topleft, *common)
    if live:
        ref_gs.tile_based_vol_rendering_scalar_backward(m2, c2, dp, al, start, end, rids, rso, rgm, rgc, rgs, rga, gso,
                                                        topleft, *common)
    torch.cuda.synchronize()
    for a_, b_, n_ in ((gm, rgm, "s g_mean2d"), (gc, rgc, "s g_cov2d"), (gs_, rgs, "s g_scalar"), (ga, rga, "s g_alpha")):
        R.grad(n_, a_, b_)
    # K9 / K10 at the scene's SH degree (c1: C=1, c2: C=3), c2w passed as the [3,4] tensor like sh_renderer.py:324
    C = sc.C
    sh = sc.sh[mask].contiguous()
    o, ro = torch.zeros(H * W * 3, device=DEV), torch.zeros(H * W * 3, device=DEV)
    _backend.tile_based_vol_rendering_sh(m2, c2, sh, al, start, end, rids, o, topleft, c2w, *common[:7], C, 1e-4)
    if live:
        ref_gs.tile_based_vol_rendering_sh(m2, c2, sh, al, start, end, rids, ro, topleft, c2w, *common[:7], C, 1e-4)
    torch.cuda.synchronize()
    shc, c2wc = sh.cpu(), c2w.cpu()
    sh_margin = lambda: oracle_mod.composite_sh_fwd(cpu[0], cpu[1], shc, cpu[2], cpu[3], cpu[4], cpu[5], cpu[6], c2wc,
                                                    C, cfg_o, want_margin=True)[3]

    def sh_exact():
        e, _, mx = oracle_mod.composite_sh_fwd_exact(cpu[0], cpu[1], shc, cpu[2], cpu[3], cpu[4], cpu[5], cpu[6], c2wc,
                                                     C, cfg_o)
        return e, mx

    close(f"sh rgb C={C}", o.view(H, W, 3), ro.view(H, W, 3), margin_fn=sh_margin, exact_fn=sh_exact)
    gm, gc, gsh, ga = torch.zeros_like(m2), torch.zeros_like(c2), torch.zeros_like(sh), torch.zeros_like(al)
    rgm, rgc, rgsh, rga = torch.zeros_like(m2), torch.zeros_like(c2), torch.zeros_like(sh), torch.zeros_like(al)
    go = gout.view(-1).contiguous()
    _backend.tile_based_vol_rendering_backward_sh(m2, c2, sh, al, start, end, rids, ro if live else o, gm, gc, gsh, ga,
                                                  go, topleft, c2w, *common[:7], C, 1e-4)
    if live:
        ref_gs.tile_based_vol_rendering_backward_sh(m2, c2, sh, al, start, end, rids, ro, rgm, rgc, rgsh, rga, go,
                                                    topleft, c2w, *common[:7], C, 1e-4)
    torch.cuda.synchronize()
    for a_, b_, n_ in ((gm, rgm, "sh g_mean2d"), (gc, rgc, "sh g_cov2d"), (gsh, rgsh, "g_sh"), (ga, rga, "sh g_alpha")):
        R.grad(n_, a_, b_)
    R.save()
