"""gsb200_estimate_normals / _backward on the B200 against the g++ host build of the same per-point math
(tests/hostmath/normals_host.cpp) and the float64 torch reference of tests/test_normals_cpu.py; the renderer's
`normal_as_rgb` batch and a relight loop on the CUDA path."""
import math

import pytest
import torch
import torch.nn.functional as F

from gsgen_b200.normals import compute_shaded_color, estimate_normal
from tests.test_normals_cpu import (_backward_reference64, host_normals, host_normals_backward, make_cloud,
                                    normals_host)  # noqa: F401  (normals_host: the fixture)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _cuda_normals(pts, K, disambiguate=True):
    """(normals, neighbour indices int32 [N,K]) through the autograd Function (indices saved for the backward)"""
    p = pts.to(DEV).requires_grad_()
    n = estimate_normal(p, K, disambiguate)
    nbr = n.grad_fn.saved_tensors[1]
    return p, n, nbr


@pytest.mark.parametrize("K", [10, 30, 50, 64])
@pytest.mark.parametrize("cloud", ["plane", "sphere", "blob", "coincident"])
def test_cuda_matches_host_build(normals_host, cloud, K):
    pts = make_cloud(cloud, n=20000, seed=5)
    nh, nbrh, _, _ = host_normals(normals_host, pts, K)
    _, n, nbr = _cuda_normals(pts, K)
    assert torch.equal(nbr.cpu(), nbrh), "neighbour indices differ"
    err = (n.detach().cpu() - nh).abs().max().item()
    assert err <= 1e-6, err  # same fp32 operations in the same order (-fmad=false): expected bit-exact
    print(f"normals {cloud} K={K}: max |cuda - host| = {err:.3g}")


def test_one_million_points_sampled_against_float64(oracle_mod):
    """1 M points on a noisy sphere shell, K = 30: 512 sampled rows meet the float64 criteria of test_normals_cpu"""
    g = torch.Generator().manual_seed(0)
    v = torch.randn(1_000_000, 3, generator=g)
    pts = v / v.norm(dim=1, keepdim=True) * (1 + 0.01 * torch.randn(1_000_000, 1, generator=g))
    K = 30
    _, n, nbr = _cuda_normals(pts, K)
    n = n.detach().cpu().double()
    rows = torch.randperm(pts.shape[0], generator=g)[:512]
    _, idx = oracle_mod.knn_points(pts[rows], pts, K)
    assert torch.equal(nbr.cpu()[rows].long(), idx)
    d = pts[idx].double() - pts[rows].double()[:, None, :]
    e = d - d.mean(1, keepdim=True)
    lam, vec = torch.linalg.eigh((e[..., :, None] * e[..., None, :]).mean(1))
    ref = vec[..., 0]
    proj = (d * ref[:, None, :]).sum(-1)
    n_pos = (proj > 0).sum(1)
    ref = torch.where((2 * n_pos < K)[:, None], -ref, ref)
    cos = (n[rows] * ref).sum(1)
    gap_ok = (lam[:, 1] - lam[:, 0]) >= 1e-3 * lam[:, 2]
    assert gap_ok.float().mean() > 0.9
    ang = torch.acos(cos.abs().clamp(max=1.0))
    assert ang[gap_ok].max() <= 1e-3, ang[gap_ok].max()
    apart = (d != 0).any(-1)
    min_rel = torch.where(apart, proj.abs(), math.inf).amin(1) / d.norm(dim=-1).amax(1)
    sign_ok = gap_ok & ((n_pos.double() - K / 2).abs() >= 1) & (min_rel >= 1e-6)
    assert sign_ok.float().mean() > 0.5 and (cos[sign_ok] > 0).all()
    assert torch.isfinite(n).all()


def test_forward_is_deterministic():
    pts = make_cloud("blob", n=200000, seed=9).to(DEV)
    a = estimate_normal(pts, 30)
    b = estimate_normal(pts, 30)
    assert torch.equal(a, b)


@pytest.mark.parametrize("cloud,K", [("plane", 10), ("plane", 30), ("cylinder", 16), ("sphere", 50), ("plane", 64)])
def test_backward_matches_float64(normals_host, cloud, K):
    pts = make_cloud(cloud, n=20000, seed=7)
    p, n, nbr = _cuda_normals(pts, K)
    g = torch.randn(pts.shape[0], 3, generator=torch.Generator().manual_seed(1))
    (n * g.to(DEV)).sum().backward()
    ref = _backward_reference64(pts, nbr.cpu().long(), n.detach().cpu(), g, True)
    rel = ((p.grad.cpu().double() - ref).norm() / ref.norm()).item()
    assert rel <= 1e-3, rel
    host = host_normals_backward(normals_host, pts, K, True, nbr.cpu(), g)
    assert ((p.grad.cpu() - host).norm() / host.norm()).item() <= 1e-5
    print(f"normals backward {cloud} K={K}: rel l2 vs float64 {rel:.3g}")


def test_errors():
    pts = make_cloud("blob", n=100).to(DEV)
    with pytest.raises(RuntimeError):
        estimate_normal(pts, 65)
    with pytest.raises(RuntimeError):
        estimate_normal(pts[:20], 30)
    from gsgen_b200 import _lib
    import ctypes

    out = torch.empty(20, 3, device=DEV)
    for K in (65, 30):  # the C ABI checks on its own
        rc = _lib.lib().gsb200_estimate_normals(_lib.ctx(DEV), _lib.fptr(pts[:20].contiguous()), ctypes.c_uint32(20),
                                                ctypes.c_int32(K), ctypes.c_int32(1), _lib.fptr(out), None,
                                                _lib.stream_ptr(DEV))
        assert rc != 0


def _scene_renderer(cfg):
    from gsgen_b200.scenes import make_scene
    from gsgen_b200.splatting import GaussianSplattingRenderer

    sc = make_scene("c3", N=20000, reso=128)
    init = {"mean": sc.mean, "qvec": sc.qvec, "svec": sc.svec * 3.0, "color": sc.color.clamp(0.05, 0.95),
            "alpha": sc.alpha}
    return GaussianSplattingRenderer(cfg, init, device=DEV), sc


def test_renderer_normal_as_rgb_on_the_gpu():
    cfg = {"normal_as_rgb": True, "normal": {"neighborhood_size": 30, "disambiguate_directions": True}}
    r, sc = _scene_renderer(cfg)
    c2w2 = sc.c2ws[0].clone()
    c2w2[:3, 3] += torch.tensor([0.05, -0.03, 0.02], device=c2w2.device)  # a second, slightly moved view
    batch = {"c2w": torch.stack([sc.c2ws[0], c2w2]), "camera_info": [sc.cams[0], sc.cams[0]]}
    r.store.zero_grad()
    out = r(batch, use_bg=False, rgb_only=True)
    out["rgb"].square().mean().backward()
    g_mean, g_color = r.store.grad_views["mean"].clone(), r.store.grad_views["color"].clone()
    r.post_backward()
    r2, _ = _scene_renderer(cfg)
    r2.store.zero_grad()
    n = estimate_normal(r2.mean, 30, True)
    views = [r2.render_one(batch["c2w"][i], batch["camera_info"][i], False, True, overrides={"color": (n + 1) / 2})
             for i in range(len(batch["camera_info"]))]
    rgb = (F.normalize(torch.stack([v["rgb"] for v in views]), dim=-1, eps=1e-6) + 1) / 2
    err = (out["rgb"] - rgb).abs().max().item()
    assert err <= 1e-4, err
    rgb.square().mean().backward()
    r2.post_backward()
    g2 = r2.store.grad_views["mean"]
    assert g_color.abs().sum() == 0 and g_mean.abs().sum() > 0
    rel = ((g_mean - g2).norm() / g2.norm()).item()
    assert rel <= 1e-3, rel
    print(f"normal_as_rgb on the GPU: image {err:.3g}, mean gradient rel l2 {rel:.3g}")


def test_relight_loop():
    """utils/relight.py's loop: K = 10 normals, compute_shaded_color per light, render_one(overrides, rgb_only)"""
    r, sc = _scene_renderer({})
    r.eval()
    c2w, cam = sc.c2ws[0], sc.cams[0]
    with torch.no_grad():
        normal = estimate_normal(r.mean.data, neighborhood_size=10)
        light_color = torch.tensor([1.0, 1.0, 1.0], device=DEV)
        az = torch.linspace(0, 2 * math.pi, 4)
        lights = torch.stack([torch.cos(az) * 3, torch.sin(az) * 3, torch.ones_like(az) * 3], -1).to(DEV)
        cam_pos = c2w[:3, 3].to(DEV)
        for lp in lights:
            color = compute_shaded_color(lp, light_color, normal, r.color.data, r.mean.data, cam_pos)
            direct = ((F.normalize(F.normalize(lp - r.mean, dim=-1) + F.normalize(cam_pos - r.mean, dim=-1), dim=-1)
                       * normal).sum(-1).abs().clamp(0, 1))[:, None] * r.color
            assert torch.allclose(color, direct, atol=1e-6)
            img = r.render_one(c2w, cam, overrides={"color": color}, rgb_only=True)["rgb"]
            assert torch.isfinite(img).all() and img.shape[-1] == 3
