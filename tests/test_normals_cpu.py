"""Normal estimation (gsgen_b200/normals.py, csrc/normals.cuh) without a GPU.

* The kernels' per-point math, built for the host with g++ over the same grid search (tests/hostmath/normals_host.cpp),
  against a float64 torch reference on brute-force neighbours (`normals_from_neighbors` on `oracle.knn_points`,
  `torch.linalg.eigh`): neighbour indices bit-exact; normals within 1e-3 rad wherever the relative eigen gap
  (lam1 - lam0) / lam2 >= 1e-3; the sign equal wherever the disambiguation count is >= 1 away from K/2 and no
  projection is below 1e-6 of the neighbourhood's extent; degenerate neighbourhoods give finite unit vectors.
* The backward formula (eigenvector perturbation through the covariance, sign held) against float64 autograd through
  `eigh` on well-gapped clouds.
* The renderer's `normal_as_rgb` path (oracle as `render_fn`, brute force as `knn_fn`) against the hand-composed
  reference expression, and bit-identical output with the flag off.
* `compute_shaded_color` / `angle_bisector` against the values the reference's own functions produced."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest
import torch

from gsgen_b200.normals import angle_bisector, compute_shaded_color, estimate_normal, normals_from_neighbors
from tests.util import GOLDEN

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KS = [1, 3, 10, 30, 50, 64]


@pytest.fixture(scope="module")
def normals_host():
    """g++ build of normals.cuh + knn_grid.cuh (rebuilt when a header or the source is newer than the library)"""
    d = os.path.join(ROOT, "tests", "hostmath")
    so = os.path.join(d, "libnormals_host.so")
    src = os.path.join(d, "normals_host.cpp")
    hdrs = [os.path.join(ROOT, "gsgen_b200", "csrc", h) for h in ("gsb200_math.cuh", "knn_grid.cuh", "normals.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(f) for f in [src] + hdrs):
        subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src,
                               "-o", so])
    return ctypes.CDLL(so)


def _vp(t):
    return ctypes.c_void_p(t.data_ptr())


def host_normals(lib, pts, K, disambiguate=True):
    n = pts.shape[0]
    pts = pts.to(torch.float32).contiguous()
    nrm = torch.empty(n, 3)
    nbr = torch.empty(n, K, dtype=torch.int32)
    lam = torch.empty(n, 3)
    deg = torch.empty(n, dtype=torch.int32)
    rc = lib.hn_normals(n, _vp(pts), K, int(disambiguate), _vp(nrm), _vp(nbr), _vp(lam), _vp(deg))
    assert rc == 0
    return nrm, nbr, lam, deg.bool()


def host_normals_backward(lib, pts, K, disambiguate, nbr, g):
    pts = pts.to(torch.float32).contiguous()
    grad = torch.zeros_like(pts)
    rc = lib.hn_normals_backward(pts.shape[0], _vp(pts), K, int(disambiguate), _vp(nbr.contiguous()),
                                 _vp(g.to(torch.float32).contiguous()), _vp(grad))
    assert rc == 0
    return grad


def make_cloud(name, n=1500, seed=0):
    g = torch.Generator().manual_seed(seed)
    if name == "plane":
        xy = torch.rand(n, 2, generator=g) * 2 - 1
        p = torch.cat([xy, 0.01 * torch.randn(n, 1, generator=g)], 1)
        R = torch.linalg.qr(torch.randn(3, 3, generator=g))[0]  # a tilted plane
        return p @ R.T + torch.tensor([3.0, -2.0, 1.0])
    if name == "sphere":
        v = torch.randn(n, 3, generator=g)
        return v / v.norm(dim=1, keepdim=True) * (1 + 0.002 * torch.randn(n, 1, generator=g))
    if name == "cylinder":
        a = torch.rand(n, generator=g) * 2 * math.pi
        return torch.stack([torch.cos(a), torch.sin(a), torch.rand(n, generator=g) * 4 - 2], 1)
    if name == "blob":
        return torch.randn(n, 3, generator=g)
    if name == "coincident":
        return torch.cat([torch.full((300, 3), 0.25), torch.randn(n - 300, 3, generator=g)])
    if name == "lattice":
        m = round(n ** (1 / 3))
        ax = torch.arange(m, dtype=torch.float32) * 0.1
        return torch.stack(torch.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(-1, 3)
    raise KeyError(name)


CLOUDS = ["plane", "sphere", "cylinder", "blob", "coincident", "lattice"]


def reference64(pts, idx, disambiguate=True):
    """float64 normals, eigenvalues, the disambiguation count and the smallest |projection| / extent per point (over
    the neighbours not at the point itself)"""
    p = pts.double()
    n = normals_from_neighbors(p, idx, disambiguate)
    d = p[idx] - p[:, None, :]
    e = d - d.mean(1, keepdim=True)
    lam = torch.linalg.eigvalsh((e[..., :, None] * e[..., None, :]).mean(1))
    proj = (d * n[:, None, :]).sum(-1)
    n_pos = (proj > 0).sum(1)
    extent = d.norm(dim=-1).amax(1)
    # (a neighbour at the point itself projects to exactly 0 in every precision: it cannot make the counts differ)
    apart = (d != 0).any(-1)
    min_rel_proj = torch.where(apart, proj.abs(), math.inf).amin(1) / extent.clamp_min(1e-300)
    return n, lam, n_pos, min_rel_proj


def check_against_reference(nrm, nbr, pts, K, idx_ref, what):
    """the criteria of the module docstring; returns (rows with a well-defined direction, rows with a defined sign)"""
    assert torch.equal(nbr.long(), idx_ref), f"{what}: neighbour indices differ"
    assert torch.isfinite(nrm).all(), what
    assert torch.allclose(nrm.double().norm(dim=1), torch.ones(nrm.shape[0], dtype=torch.float64), atol=1e-5), what
    n64, lam, n_pos, min_rel_proj = reference64(pts, idx_ref)
    gap_ok = (lam[:, 1] - lam[:, 0]) >= 1e-3 * lam[:, 2]
    cos = (nrm.double() * n64).sum(1)
    ang = torch.acos(cos.abs().clamp(max=1.0))
    if gap_ok.any():
        worst = ang[gap_ok].max().item()
        assert worst <= 1e-3, f"{what}: angle {worst:.3g} rad"
    sign_ok = gap_ok & ((n_pos.double() - K / 2).abs() >= 1) & (min_rel_proj >= 1e-6)
    assert (cos[sign_ok] > 0).all(), f"{what}: {(cos[sign_ok] <= 0).sum().item()} signs differ"
    return int(gap_ok.sum()), int(sign_ok.sum())


@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("cloud", CLOUDS)
def test_host_normals_match_float64_reference(normals_host, oracle_mod, cloud, K):
    pts = make_cloud(cloud)
    nrm, nbr, lam, deg = host_normals(normals_host, pts, K)
    _, idx_ref = oracle_mod.knn_points(None, pts, K)
    n_gap, n_sign = check_against_reference(nrm, nbr, pts, K, idx_ref, f"{cloud} K={K}")
    if K == 1:
        # a lone point has a zero covariance: (0, 0, 1), flipped (no neighbour lies strictly on its positive side)
        assert deg.all() and torch.equal(nrm, torch.tensor([0.0, 0.0, -1.0]).expand_as(nrm))
    if cloud == "coincident" and K > 1:
        assert deg[:300].all()  # (the 300 copies are each other's nearest neighbours, ties by index)
    if cloud in ("plane", "sphere", "cylinder") and K >= 10:
        assert n_gap > 0.9 * pts.shape[0] and n_sign > 0.5 * pts.shape[0], (n_gap, n_sign)


def test_plane_normals_and_orientation(normals_host):
    """on a plane every normal is the plane's (up to sign), and the sign rule picks the side with more neighbours"""
    pts = make_cloud("plane", n=2000, seed=3)
    nrm, _, _, deg = host_normals(normals_host, pts, 30)
    assert not deg.any()
    c = pts - pts.mean(0)
    axis = torch.linalg.eigh(c.T @ c)[1][:, 0]
    assert (nrm @ axis).abs().min() > 0.99


@pytest.mark.parametrize("K", [10, 30, 64])
def test_disambiguation_off_gives_the_same_axis(normals_host, K):
    pts = make_cloud("sphere", seed=4)
    a, _, _, _ = host_normals(normals_host, pts, K, True)
    b, _, _, _ = host_normals(normals_host, pts, K, False)
    assert torch.equal(a.abs(), b.abs())


def test_host_errors(normals_host):
    pts = make_cloud("blob", n=40).contiguous()
    out = torch.empty(40, 3)
    nbr = torch.empty(40, 65, dtype=torch.int32)
    lam, deg = torch.empty(40, 3), torch.empty(40, dtype=torch.int32)
    assert normals_host.hn_normals(40, _vp(pts), 65, 1, _vp(out), _vp(nbr), _vp(lam), _vp(deg)) == 1
    assert normals_host.hn_normals(40, _vp(pts), 41, 1, _vp(out), _vp(nbr), _vp(lam), _vp(deg)) == 1
    with pytest.raises(RuntimeError):
        estimate_normal(pts, neighborhood_size=65)
    with pytest.raises(RuntimeError):
        estimate_normal(pts, neighborhood_size=41)
    with pytest.raises(RuntimeError, match="CUDA"):
        estimate_normal(pts, neighborhood_size=10)  # no CPU fallback without a `knn=` search


def _backward_reference64(pts, idx, nrm_host, g, disambiguate):
    """float64 autograd through eigh, with the host's signs (the sign is piecewise constant, held in both)"""
    p = pts.double().clone().requires_grad_()
    n = normals_from_neighbors(p, idx, False)
    s = torch.sign((n.detach() * nrm_host.double()).sum(1, keepdim=True))
    ((s * n) * g.double()).sum().backward()
    return p.grad


@pytest.mark.parametrize("cloud,K", [("plane", 10), ("plane", 30), ("cylinder", 16), ("sphere", 50), ("plane", 64)])
def test_backward_matches_float64_autograd(normals_host, oracle_mod, cloud, K):
    pts = make_cloud(cloud, n=1200, seed=7)
    nrm, nbr, lam, deg = host_normals(normals_host, pts, K)
    assert not deg.any()
    # well gapped: the smallest eigenvalue is separated from the other two
    assert ((lam[:, 1] - lam[:, 0]) / lam[:, 2]).min() > 1e-2
    g = torch.randn(pts.shape[0], 3, generator=torch.Generator().manual_seed(1))
    ours = host_normals_backward(normals_host, pts, K, True, nbr, g)
    ref = _backward_reference64(pts, nbr.long(), nrm, g, True)
    rel = ((ours.double() - ref).norm() / ref.norm()).item()
    assert rel <= 1e-4, rel


def test_backward_zero_for_degenerate_and_isotropic_patches(normals_host):
    """coincident neighbourhoods and a lattice's isotropic ones (equal eigenvalues): finite, and zero where every gap is
    below the guard"""
    pts = make_cloud("coincident", n=600)
    nrm, nbr, _, deg = host_normals(normals_host, pts, 10)
    g = torch.zeros(600, 3)
    g[:300] = 1.0  # gradient only on the degenerate rows
    grad = host_normals_backward(normals_host, pts, 10, True, nbr, g)
    assert deg[:300].all() and torch.equal(grad, torch.zeros_like(grad))
    lat = make_cloud("lattice", n=1000)
    nrm, nbr, lam, deg = host_normals(normals_host, lat, 7)  # centre + its 6 axis neighbours: lam0 = lam1 = lam2
    interior = ((lat > 0.05) & (lat < 0.85)).all(1)
    assert ((lam[interior, 2] - lam[interior, 0]).abs() <= 1e-6 * lam[interior, 2]).all()
    g = torch.zeros_like(lat)
    g[interior] = 1.0
    grad = host_normals_backward(normals_host, lat, 7, True, nbr, g)
    assert torch.isfinite(grad).all() and torch.equal(grad, torch.zeros_like(grad))


def test_torch_path_autograd_and_knn_hook(oracle_mod):
    """estimate_normal(knn=...) is the torch composition on the hook's neighbours; gradients reach the points"""
    pts = make_cloud("plane", n=400, seed=2).requires_grad_()
    n = estimate_normal(pts, 20, True, knn=oracle_mod.knn_points)
    _, idx = oracle_mod.knn_points(None, pts, 20)
    assert torch.equal(n, normals_from_neighbors(pts, idx, True))
    n.sum().backward()
    assert torch.isfinite(pts.grad).all() and pts.grad.abs().sum() > 0


# ---- renderer ---------------------------------------------------------------------------------------------------
def _render_fn(oracle_mod):
    """the oracle on raw leaves or on activated values (render_one(overrides=...) renders the latter)"""
    from tests.test_splatting_cpu import _Aux, ocam_of

    def fn(mean, qvec, svec, alpha, c2w, cam, color=None, bg=None, rgb_only=False, raw_params=False, grad_sink=None,
           slot=0, frustum_radius=6.0, tile_radius=6.0, T_thresh=1e-4, skip_frustum_culling=False, depth_detach=True):
        s, a, c = (torch.exp(svec), torch.sigmoid(alpha), torch.sigmoid(color)) if raw_params else (svec, alpha, color)
        out = oracle_mod.render_view(mean, qvec, s, a, c2w, ocam_of(cam), color=c, bg=bg, rgb_only=rgb_only,
                                     depth_detach=depth_detach, frustum_radius=frustum_radius, tile_radius=tile_radius,
                                     thresh=T_thresh)
        au = out["aux"]
        out["aux"] = _Aux(mask=au["mask"], mean2d_masked=au["mean2d"], radii2d=torch.zeros(mean.shape[0]),
                          N_with_dub=au["D"])
        out.setdefault("T", None)
        return out

    return fn


def _renderer(oracle_mod, cfg):
    from gsgen_b200.scenes import make_scene
    from gsgen_b200.splatting import GaussianSplattingRenderer

    sc = make_scene("c1", N=300, reso=48)
    init = {"mean": sc.mean, "qvec": sc.qvec, "svec": sc.svec * 3.0, "color": sc.color.clamp(0.05, 0.95),
            "alpha": sc.alpha}
    r = GaussianSplattingRenderer(cfg, init, device="cpu", render_fn=_render_fn(oracle_mod),
                                  knn_fn=oracle_mod.knn_points)
    return r, sc


def test_renderer_normal_as_rgb_matches_composition(oracle_mod):
    import torch.nn.functional as F

    cfg = {"normal_as_rgb": True, "normal": {"neighborhood_size": 30, "disambiguate_directions": True}}
    r, sc = _renderer(oracle_mod, cfg)
    c2w2 = sc.c2ws[0].clone()
    c2w2[:3, 3] += torch.tensor([0.05, -0.03, 0.02])  # a second, slightly moved view
    batch = {"c2w": torch.stack([sc.c2ws[0], c2w2]), "camera_info": [sc.cams[0], sc.cams[0]]}
    out = r(batch, use_bg=False, rgb_only=True)
    loss = out["rgb"].square().mean()
    loss.backward()
    g_color = r.store.grad_views["color"].clone()
    g_mean_leaf = r.store.params["mean"].grad
    # hand-composed: the reference's forward with the normal estimated once for the batch
    r2, _ = _renderer(oracle_mod, cfg)
    n = estimate_normal(r2.mean, 30, True, knn=oracle_mod.knn_points)
    views = [r2.render_one(batch["c2w"][i], batch["camera_info"][i], False, True, overrides={"color": (n + 1) / 2})
             for i in range(2)]
    rgb = (F.normalize(torch.stack([v["rgb"] for v in views]), dim=-1, eps=1e-6) + 1) / 2
    # (the views run on the raw leaves with the colour as logit((n + 1) / 2): the sigmoid gives it back to rounding)
    assert (out["rgb"] - rgb).abs().max() <= 1e-5
    assert torch.equal(r.normal, n.detach())
    # the colour leaves do not take part; the means get a gradient through the normals (and the projection)
    assert g_color.abs().sum() == 0
    assert g_mean_leaf is not None and g_mean_leaf.abs().sum() > 0
    rgb.square().mean().backward()
    g1, g2 = r.store.grad_views["mean"], r2.store.grad_views["mean"]
    assert ((g1 - g2).norm() / g2.norm()) <= 1e-4


def test_renderer_normal_as_rgb_off_is_unchanged(oracle_mod):
    base = {"normal": {"neighborhood_size": 30, "disambiguate_directions": True}}
    r1, sc = _renderer(oracle_mod, dict(base, normal_as_rgb=False))
    r2, _ = _renderer(oracle_mod, {})
    batch = {"c2w": sc.c2ws[0][None], "camera_info": [sc.cams[0]]}
    o1, o2 = r1(batch, use_bg=False), r2(batch, use_bg=False)
    for k in o2:
        assert torch.equal(o1[k], o2[k]), k


def test_renderer_normal_property_defaults(oracle_mod):
    """no `normal` block: estimate_normal's own defaults (50 neighbours, disambiguated); update_normal does not raise"""
    r, _ = _renderer(oracle_mod, {})
    n = r.update_normal()
    assert torch.equal(n, estimate_normal(r.mean, 50, True, knn=oracle_mod.knn_points))


# ---- shading --------------------------------------------------------------------------------------------------------
def test_compute_shaded_color_matches_reference_values():
    z = np.load(os.path.join(GOLDEN, "shaded_color_ref.npz"))
    t = {k: torch.from_numpy(z[k]) for k in z.files}
    for i in range(t["lights"].shape[0]):
        lp, lc = t["lights"][i], t["light_colors"][i]
        got = compute_shaded_color(lp, lc, t["normal"], t["color"], t["mean"], t["cam_pos"])
        assert torch.equal(got, t["shaded"][i]), i
        assert torch.equal(angle_bisector(lp - t["mean"], t["cam_pos"] - t["mean"]), t["bisector"][i]), i
