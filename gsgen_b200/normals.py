"""Point-cloud normals of the Gaussian means and the shading helpers built on them -- the host-side mirror of
`utils/ops.py:58-72` (`angle_bisector`, `estimate_normal`) and `:188-195` (`compute_shaded_color`) over
`gsb200_estimate_normals` (csrc/normals.cu: grid neighbour search + per-point PCA fused in one kernel).

`estimate_normal` sits on `pytorch3d.ops.estimate_pointcloud_normals` in the reference (third party, optional import,
unpinned, absent in this image, so this could not be checked against the library).  Its contract as restated here:
  * neighbourhood: `knn_points(p, p, K)` -- the K nearest points, the point itself included (ties by point index);
  * covariance: the mean over K of (x_k - mu)(x_k - mu)^T, mu the neighbourhood mean;
  * normal: the unit eigenvector of the smallest eigenvalue;
  * disambiguation (`disambiguate_directions`): with proj_k = n . (x_k - p) measured from the point p itself, n is
    negated when fewer than K/2 of the proj_k are > 0.
Ours, where pytorch3d leaves the case undefined: fewer points than K raises; a zero covariance (coincident neighbours,
K = 1) gives (0, 0, 1) before the flip and no gradient.

Gradients reach the points through the covariance with the neighbour sets and the sign held constant (as autograd
through pytorch3d's `knn_gather` and its piecewise-constant flip).  One deliberate difference from autograd through
`torch.linalg.eigh`: an eigen gap |lam_0 - lam_j| <= 1e-6 max(lam_2, 1e-30) contributes zero instead of inf / NaN, so a
flat or isotropic patch cannot poison the gradient arena.

CUDA tensors only -- there is no CPU fallback.  `knn=` (a `knn_points`-style search, e.g. the oracle's brute force)
switches to the same math composed from torch ops; the CPU test-suite uses that path, and it is the reference the
kernel is tested against."""
from __future__ import annotations

import ctypes
from typing import Callable, Optional

import torch
import torch.nn.functional as F

from . import _lib

MAX_K = 64


def angle_bisector(a, b):
    """utils/ops.py:58-59"""
    return F.normalize(F.normalize(a, dim=-1) + F.normalize(b, dim=-1), dim=-1)


def compute_shaded_color(light_pos, light_color, surface_normal, surface_color, mean, cam_pos):
    """utils/ops.py:188-195 (= `compute_color` of utils/relight.py:13-18): |cos| of the angle between the normal and the
    bisector of the directions to the light and to the camera (two-sided), times light and surface colour"""
    ab = angle_bisector(light_pos - mean, cam_pos - mean)
    # backface culling
    dot = (ab * surface_normal).sum(dim=-1).abs().clamp(min=0.0, max=1.0)

    return light_color * dot[..., None] * surface_color


def _check(pos: torch.Tensor, K: int):
    if pos.dim() != 2 or pos.shape[1] != 3:
        raise RuntimeError(f"pos must be [N,3], got {tuple(pos.shape)}")
    if not 1 <= int(K) <= MAX_K:
        raise RuntimeError(f"neighborhood_size = {K} outside [1, {MAX_K}]")
    if pos.shape[0] < int(K):
        raise RuntimeError(f"neighborhood_size = {K} needs at least {K} points, got {pos.shape[0]}")


class _EstimateNormals(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, K: int, disambiguate: bool):
        dev = pos.device
        pts = pos.detach().to(torch.float32).contiguous()
        n = pts.shape[0]
        normals = torch.empty(n, 3, dtype=torch.float32, device=dev)
        nbr = torch.empty(n, K, dtype=torch.int32, device=dev) if ctx.needs_input_grad[0] else None
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().gsb200_estimate_normals(
                _lib.ctx(dev), _lib.fptr(pts, "pos"), ctypes.c_uint32(n), ctypes.c_int32(K),
                ctypes.c_int32(int(disambiguate)), _lib.fptr(normals, "normals"), _lib.ptr(nbr, torch.int32, "nbr"),
                _lib.stream_ptr(dev)))
        ctx.K, ctx.disambiguate, ctx.dtype = K, disambiguate, pos.dtype
        ctx.save_for_backward(pts, nbr)
        return normals

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_normals):
        pts, nbr = ctx.saved_tensors
        dev = pts.device
        g = grad_normals.to(torch.float32).contiguous()
        grad = torch.zeros_like(pts)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().gsb200_estimate_normals_backward(
                _lib.ctx(dev), _lib.fptr(pts, "pos"), ctypes.c_uint32(pts.shape[0]), ctypes.c_int32(ctx.K),
                ctypes.c_int32(int(ctx.disambiguate)), _lib.ptr(nbr, torch.int32, "nbr"), _lib.fptr(g, "grad_normals"),
                _lib.fptr(grad, "grad_pos"), _lib.stream_ptr(dev)))
        return grad.to(ctx.dtype), None, None


def normals_from_neighbors(pos: torch.Tensor, idx: torch.Tensor, disambiguate_directions: bool = True) -> torch.Tensor:
    """The per-point math of the kernel composed from torch ops, for given neighbour indices idx [N,K] (the point
    itself included): covariance relative to the point, `torch.linalg.eigh`, smallest eigenvector, sign rule,
    (0, 0, 1) for a zero covariance.  Differentiable (through eigh: no gap guard); works in pos's dtype."""
    K = idx.shape[1]
    d = pos[idx] - pos[:, None, :]                                   # x_k - p  [N,K,3]
    e = d - d.mean(dim=1, keepdim=True)
    cov = (e[..., :, None] * e[..., None, :]).mean(dim=1)            # [N,3,3]
    degenerate = ~((cov.detach().abs().amax(dim=(-2, -1)) > 0) & torch.isfinite(cov.detach()).all(-1).all(-1))
    safe = torch.where(degenerate[:, None, None], torch.diag(torch.tensor([1.0, 2.0, 3.0], dtype=pos.dtype,
                                                                          device=pos.device)), cov)
    _, vecs = torch.linalg.eigh(safe)
    n = vecs[..., 0]
    up = torch.tensor([0.0, 0.0, 1.0], dtype=pos.dtype, device=pos.device).expand_as(n)
    n = torch.where(degenerate[:, None], up, n)
    if disambiguate_directions:
        proj = (d.detach() * n.detach()[:, None, :]).sum(-1)
        flip = 2 * (proj > 0).sum(dim=1) < K
        n = torch.where(flip[:, None], -n, n)
    return n


def estimate_normal(pos: torch.Tensor, neighborhood_size: int = 50, disambiguate_directions: bool = True,
                    knn: Optional[Callable] = None) -> torch.Tensor:
    """utils/ops.py:62-72: one unit normal per point of pos [N,3] (see the module docstring) -> [N,3] fp32.
    `knn`: a `knn_points(query, points, K, return_dist)` search; given, the torch composition above runs instead of the
    kernel (its result has pos's dtype)."""
    K = int(neighborhood_size)
    _check(pos, K)
    if knn is not None:
        _, idx = knn(None, pos, K, False)
        return normals_from_neighbors(pos, idx.to(pos.device), bool(disambiguate_directions))
    if not pos.is_cuda:
        raise RuntimeError("gsgen_b200.normals needs CUDA tensors (libgsb200 has no CPU path)")
    return _EstimateNormals.apply(pos, K, bool(disambiguate_directions))
